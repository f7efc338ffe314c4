// tinybvh_b200/csrc/build_hq.cu - SBVH construction (spatial splits) on sm_100a.
//
// Replaces BVH::BuildHQ: PrepareHQBuild (tiny_bvh.h:2648-2709), BuildHQTask (:2731-3008), SplitCostSAH (:2711), ClipFrag
// (:8614-8729), SplitFrag (:8731-8793) and the closing Compact() (:3733-3770).  The result is the reference's own tree
// byte for byte (tests/test_build_hq_gpu.py memcmp()s nodes and the referenced part of primIdx against it), which pins
// down more than the split decisions:
//   * every float operation is spelled with an _rn intrinsic in the pairing of the frozen reference build (see the
//     header of oracle/tbvh_oracle_hq.c); nvcc's own contraction cannot change a rounding;
//   * the "unsplitting" pass (:2895-2926) is a sequential chain over the straddling fragments of a node - each decision
//     changes the running child bounds / counts / cost the next one is judged by.  Here the fragments of a node are
//     classified in parallel, the straddlers are compacted in order, ONE warp walks the chain (32 straddlers fetched per
//     step, decisions replayed from registers), and the fragments the chain decides to split are clipped in parallel;
//   * the reference partitions into a second index array (idxTmp) inside the node's slice [sliceStart, sliceEnd) and, when a
//     spatial split "fails" (:2939, all fragments end up on one side), builds the leaf from whatever idxTmp held at the
//     node's old position - words written by an ancestor's partition, or the initial zeros.  That is reproduced by keeping
//     the same two arrays with the same write discipline (left part upward from sliceStart, right part downward from
//     sliceEnd, copy back to primIdx): what a failed node reads is then a function of its ancestors only, not of the order
//     nodes are processed in;
//   * node numbering after Compact() is "children of the k-th interior node in DFS preorder at 2+2k, 3+2k", leaf index
//     ranges packed in DFS leaf order: computed here from subtree sizes (one bottom-up pass with arrival counters, one
//     walk to the root per node).  New fragments are handed out by an atomic counter; their numbers never reach the output.
//
// Structure: every node is owned by one thread group for all of its steps (object bins, sweep, spatial bins with clipping,
// sweep, partition, child bounds, emit), so no step needs inter-CTA communication:
//   k_hq_level     level-synchronous, one 256-thread CTA per node with more than HQ_SMALL fragments
//   k_hq_subtrees  one warp per subtree of at most HQ_SMALL fragments, depth-first with a shared-memory task stack
#include "common.cuh"
#include <cooperative_groups.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

namespace cg = cooperative_groups;
namespace
{
#define HQBINS 8
#define HQ_SMALL 16            // switch point CTA/cluster per node -> warp per subtree: nodes of at most this many fragments
#define HQ_MAX_CLUSTER 16      // largest thread-block cluster a node of the level phase gets
#define HQ_CTA_FRAGS 512       // cluster sizing: about this many fragments per CTA of the level's largest node
#define HQ_CTA_CAP 16          // cluster sizing: 2 x (CTAs of the level) <= this x SMs, i.e. at most 8 CTAs per SM in flight
#define HQ_MLP 4               // independent index -> fragment load chains per thread in the binning loops
#define HQ_E 8                 // consecutive fragments per thread and scan tile of the partition passes (8 * 4096 fits the 16-bit packed counters)
#define HQ_BIG_THREADS 256
#define HQ_SMALL_WARPS 4
#define HQ_STACK 64

struct HQTask { uint32_t node, sliceStart, sliceEnd, depth; };
struct HQCounters
{
	uint32_t node_ptr;       // temp node records allocated (pairs from 2)
	uint32_t frag_ptr;       // nextFrag
	uint32_t next_big;       // tasks appended to the next level's list
	uint32_t next_max;       // largest fragment count among them (sizes the clusters); cleared together with next_big
	uint32_t small_roots;    // subtree roots for k_hq_subtrees
	uint32_t max_depth;
	uint32_t failed_splits;  // ":2939 spatial split failed" leaves
	uint32_t overflow;       // a task stack / fragment pool ran out (cannot happen within the reference's own bounds)
	uint32_t root_key[6];
	float root_area;
	float min_dim[3];
	unsigned long long prof[32]; // TBVH_HQ_PROFILE=1: leader-thread cycles per phase, [0..15] level phase, [16..31] subtree phase
};

struct HQArgs
{
	const float4* verts;
	float4* frag_min; float4* frag_max;       // (bmin, primIdx) / (bmax, clipped): the reference's 32-byte Fragment (:792) as two halves
	uint32_t* prim_idx; uint32_t* idx_tmp;    // both idx_cap words, the reference's primIdx / idxTmp
	uint32_t* cls; uint32_t* strad; float* spos; // partition scratch, indexed like the slices
	float4* tmp_nodes; uint32_t* parent; uint32_t* sub_int; uint32_t* sub_prims; uint32_t* arrive;
	HQTask* lvl[2]; HQTask* small;
	HQCounters* ctr;
	uint32_t n, idx_cap, node_cap, lvl_cap, profile;
	float c_trav, c_int;
};

struct GroupSmem
{
	uint32_t kmin[3][HQBINS][3], kmax[3][HQBINS][3]; // bin bounds as ordered keys
	uint32_t cntA[3][HQBINS], cntB[3][HQBINS];       // object: count / spatial: countIn, countOut
	float best[12];                                  // child bounds of the chosen split: lmin, lmax, rmin, rmax
	float splitCost;
	uint32_t bestAxis, bestPos, bestIdx;
	int spatial, bestNL, bestNR, hasObj, trySpatial, leaf;
	uint32_t wtot[8];
	uint32_t ctot[HQ_MAX_CLUSTER];
	uint32_t nstrad;
	uint32_t ckey[12];                               // child bounds of a spatial partition: lmin, lmax, rmin, rmax keys
	uint32_t lc;
};

// ---------------------------------------------------------------------------------------------- shared math
__device__ __forceinline__ float tmin( const float a, const float b ) { return a < b ? a : b; }   // tinybvh_min :432
__device__ __forceinline__ float tmax( const float a, const float b ) { return a > b ? a : b; }   // tinybvh_max :433
__device__ __forceinline__ float clampf( const float x, const float a, const float b ) { return x > a ? (x < b ? x : b) : a; }
__device__ __forceinline__ int clampi( const int x, const int a, const int b ) { return x > a ? (x < b ? x : b) : a; }
// (int)f as x86 computes it (cvttss2si): INT_MIN for NaN and anything outside int32
__device__ __forceinline__ int cvtt( const float f ) { return (f >= -2147483648.0f && f < 2147483648.0f) ? __float2int_rz( f ) : (int)0x80000000; }
// tinybvh_half_area :460 / BVHBase::SA :8477, the reference build's pairing
__device__ __forceinline__ float half_area3( const float x, const float y, const float z )
{
	return x < -BVH_FAR ? 0.0f : __fmaf_rn( z, x, __fmaf_rn( y, x, __fmul_rn( y, z ) ) );
}
// SplitCostSAH :2711 (l_quads = false)
__device__ __forceinline__ float split_cost( const float c_trav, const float c_int, const float rAparent, const float Aleft, const int Nleft, const float Aright, const int Nright )
{
	return __fmaf_rn( __fmaf_rn( __int2float_rn( Nleft ), Aleft, __fmul_rn( Aright, __int2float_rn( Nright ) ) ), __fmul_rn( c_int, rAparent ), c_trav );
}
__device__ __forceinline__ float comp( const float4 v, const uint32_t a ) { return a == 0 ? v.x : a == 1 ? v.y : v.z; }

struct Frag { float bmin[3], bmax[3]; uint32_t prim, clipped; };
__device__ __forceinline__ Frag load_frag( const HQArgs& A, const uint32_t fi )
{
	const float4 a = A.frag_min[fi], b = A.frag_max[fi];
	Frag f;
	f.bmin[0] = a.x, f.bmin[1] = a.y, f.bmin[2] = a.z, f.prim = __float_as_uint( a.w );
	f.bmax[0] = b.x, f.bmax[1] = b.y, f.bmax[2] = b.z, f.clipped = __float_as_uint( b.w );
	return f;
}
__device__ __forceinline__ void store_frag( const HQArgs& A, const uint32_t fi, const float* bmin, const float* bmax, const uint32_t prim )
{
	A.frag_min[fi] = make_float4( bmin[0], bmin[1], bmin[2], __uint_as_float( prim ) );
	A.frag_max[fi] = make_float4( bmax[0], bmax[1], bmax[2], __uint_as_float( 1u ) );
}
__device__ __forceinline__ void load_tri( const HQArgs& A, const uint32_t prim, float v[3][3] )
{
	#pragma unroll
	for (int k = 0; k < 3; k++) { const float4 p = A.verts[(size_t)prim * 3 + k]; v[k][0] = p.x, v[k][1] = p.y, v[k][2] = p.z; }
}
// C = v0 + f * (v1 - v0), compiled by the reference build as fma( f, v1 - v0, v0 ) per component
__device__ __forceinline__ void lerp3( float* C, const float* v0, const float* v1, const float f )
{
	#pragma unroll
	for (int k = 0; k < 3; k++) C[k] = __fmaf_rn( f, __fsub_rn( v1[k], v0[k] ), v0[k] );
}
__device__ __forceinline__ void cp3( float* d, const float* s ) { d[0] = s[0], d[1] = s[1], d[2] = s[2]; }

// Sutherland-Hodgman of polygon vin[0..Nin) against the slab l <= x[a] <= r, in place (result back in vin); the generic
// loops of ClipFrag (:8630-8658, tolerance eps, unclamped f) and SplitFrag (:8744-8770, eps = 0, f clamped to [0,1]).
template <bool CLAMP> __device__ __noinline__ uint32_t clip_slab( float vin[16][3], float vout[16][3], uint32_t Nin, const uint32_t a, const float l, const float r, const float eps )
{
	uint32_t Nout = 0;
	const float le = __fsub_rn( l, eps ), re = __fadd_rn( r, eps );
	for (uint32_t v = 0; v < Nin; v++)
	{
		const float* v0 = vin[v], * v1 = vin[v + 1 == Nin ? 0 : v + 1];
		const bool v0in = v0[a] >= le, v1in = v1[a] >= le;
		if (!(v0in || v1in)) continue; else if (v0in ^ v1in)
		{
			float f = __fdiv_rn( __fsub_rn( l, v0[a] ), __fsub_rn( v1[a], v0[a] ) );
			if (CLAMP) f = clampf( f, 0.0f, 1.0f );
			float C[3];
			lerp3( C, v0, v1, f ), C[a] = l, cp3( vout[Nout++], C );
		}
		if (v1in) cp3( vout[Nout++], v1 );
	}
	Nin = 0;
	for (uint32_t v = 0; v < Nout; v++)
	{
		const float* v0 = vout[v], * v1 = vout[v + 1 == Nout ? 0 : v + 1];
		const bool v0in = v0[a] <= re, v1in = v1[a] <= re;
		if (!(v0in || v1in)) continue; else if (v0in ^ v1in)
		{
			float f = __fdiv_rn( __fsub_rn( r, v0[a] ), __fsub_rn( v1[a], v0[a] ) );
			if (CLAMP) f = clampf( f, 0.0f, 1.0f );
			float C[3];
			lerp3( C, v0, v1, f ), C[a] = r, cp3( vin[Nin++], C );
		}
		if (v1in) cp3( vin[Nin++], v1 );
	}
	return Nin;
}

// BVH::ClipFrag :8614-8729: bounds of (fragment's triangle) clipped to box [bmin_in, bmax_in] ^ fragment box.
// Returns false when nothing is left; nb_min / nb_max receive the new fragment's box either way (as the reference does).
__device__ __noinline__ bool clip_frag( const HQArgs& A, const Frag& orig, float* nb_min, float* nb_max, const float* bmin_in, const float* bmax_in, const float* minDim, const uint32_t axis )
{
	float bmin[3], bmax[3], extent[3];
	#pragma unroll
	for (int a = 0; a < 3; a++) bmin[a] = tmax( bmin_in[a], orig.bmin[a] ), bmax[a] = tmin( bmax_in[a], orig.bmax[a] ), extent[a] = __fsub_rn( bmax[a], bmin[a] );
	float mn[3] = { BVH_FAR, BVH_FAR, BVH_FAR }, mx[3] = { -BVH_FAR, -BVH_FAR, -BVH_FAR };
	bool has;
	if (orig.clipped)
	{
		float vin[16][3], vout[16][3];
		{
			float t[3][3];
			load_tri( A, orig.prim, t );
			cp3( vin[0], t[0] ), cp3( vin[1], t[1] ), cp3( vin[2], t[2] );
		}
		uint32_t Nin = 3;
		#pragma unroll 1
		for (uint32_t a = 0; a < 3; a++)
		{
			const float eps = minDim[a];
			if (extent[a] > eps) Nin = clip_slab<false>( vin, vout, Nin, a, bmin[a], bmax[a], eps );
		}
		for (uint32_t i = 0; i < Nin; i++)
		{
			#pragma unroll
			for (int k = 0; k < 3; k++) mn[k] = tmin( mn[k], vin[i][k] ), mx[k] = tmax( mx[k], vin[i][k] );
		}
		has = Nin > 0;
	}
	else
	{
		// fragment never clipped before: only the two planes on the split axis matter (:8665-8724)
		has = false;
		if (extent[axis] > minDim[axis])
		{
			const float l = bmin[axis], r = bmax[axis];
			float vout[4][3], t[3][3], C[3];
			uint32_t Nout = 0;
			load_tri( A, orig.prim, t );
			const bool in0 = t[0][axis] >= l, in1 = t[1][axis] >= l, in2 = t[2][axis] >= l;
			#pragma unroll
			for (int e = 0; e < 3; e++)
			{
				const float* v0 = t[e], * v1 = t[(e + 1) % 3];
				const bool v0in = e == 0 ? in0 : e == 1 ? in1 : in2, v1in = e == 0 ? in1 : e == 1 ? in2 : in0;
				if (v0in || v1in)
				{
					if (v0in ^ v1in)
					{
						const float f = clampf( __fdiv_rn( __fsub_rn( l, v0[axis] ), __fsub_rn( v1[axis], v0[axis] ) ), 0.0f, 1.0f );
						lerp3( C, v0, v1, f ), C[axis] = l, cp3( vout[Nout++], C );
					}
					if (v1in) cp3( vout[Nout++], v1 );
				}
			}
			for (uint32_t v = 0; v < Nout; v++)
			{
				const float* v0 = vout[v], * v1 = vout[v + 1 == Nout ? 0 : v + 1];
				const bool v0in = v0[axis] <= r, v1in = v1[axis] <= r;
				if (!(v0in || v1in)) continue; else if (v0in ^ v1in)
				{
					const float f = clampf( __fdiv_rn( __fsub_rn( r, v0[axis] ), __fsub_rn( v1[axis], v0[axis] ) ), 0.0f, 1.0f );
					lerp3( C, v0, v1, f ), C[axis] = r, has = true;
					#pragma unroll
					for (int k = 0; k < 3; k++) mn[k] = tmin( mn[k], C[k] ), mx[k] = tmax( mx[k], C[k] );
				}
				if (v1in)
				{
					has = true;
					#pragma unroll
					for (int k = 0; k < 3; k++) mn[k] = tmin( mn[k], v1[k] ), mx[k] = tmax( mx[k], v1[k] );
				}
			}
		}
	}
	#pragma unroll
	for (int k = 0; k < 3; k++) nb_min[k] = tmax( mn[k], bmin[k] ), nb_max[k] = tmin( mx[k], bmax[k] );
	return has;
}

// BVH::SplitFrag :8731-8793: the fragment's polygon cut at splitPos; only the two halves' boxes are kept.
__device__ __noinline__ void split_frag( const HQArgs& A, const Frag& orig, float* lmin, float* lmax, float* rmin, float* rmax, const float* minDim,
	const uint32_t splitAxis, const float splitPos, bool& leftOK, bool& rightOK )
{
	float vin[16][3], vout[16][3];
	{
		float t[3][3];
		load_tri( A, orig.prim, t );
		cp3( vin[0], t[0] ), cp3( vin[1], t[1] ), cp3( vin[2], t[2] );
	}
	uint32_t Nin = 3, Nleft = 0, Nright = 0;
	if (orig.clipped)
		#pragma unroll 1
		for (uint32_t a = 0; a < 3; a++) if (__fsub_rn( orig.bmax[a], orig.bmin[a] ) > minDim[a])
		Nin = clip_slab<true>( vin, vout, Nin, a, orig.bmin[a], orig.bmax[a], 0.0f );
	#pragma unroll
	for (int k = 0; k < 3; k++) lmin[k] = rmin[k] = BVH_FAR, lmax[k] = rmax[k] = -BVH_FAR;
	#define ADD_L( p ) { Nleft++; for (int k_ = 0; k_ < 3; k_++) lmin[k_] = tmin( lmin[k_], (p)[k_] ), lmax[k_] = tmax( lmax[k_], (p)[k_] ); }
	#define ADD_R( p ) { Nright++; for (int k_ = 0; k_ < 3; k_++) rmin[k_] = tmin( rmin[k_], (p)[k_] ), rmax[k_] = tmax( rmax[k_], (p)[k_] ); }
	for (uint32_t v = 0; v < Nin; v++)
	{
		const float* v0 = vin[v], * v1 = vin[v + 1 == Nin ? 0 : v + 1];
		const bool v0left = v0[splitAxis] < splitPos, v1left = v1[splitAxis] < splitPos;
		if (v0left && v1left) ADD_L( v1 ) else if (!v0left && !v1left) ADD_R( v1 ) else
		{
			const float f = clampf( __fdiv_rn( __fsub_rn( splitPos, v0[splitAxis] ), __fsub_rn( v1[splitAxis], v0[splitAxis] ) ), 0.0f, 1.0f );
			float C[3];
			lerp3( C, v0, v1, f ), C[splitAxis] = splitPos;
			ADD_L( C ) ADD_R( C )
			if (v0left) ADD_R( v1 ) else ADD_L( v1 )
		}
	}
	#undef ADD_L
	#undef ADD_R
	leftOK = Nleft > 0, rightOK = Nright > 0;
}

// ---------------------------------------------------------------------------------------------- group helpers
// A node is owned by a "group": one warp (G = 32), one CTA (G = 256, nct = 1) or a thread-block cluster of nct CTAs.  In a
// cluster every CTA keeps its own GroupSmem (bins, scan scratch); the leader's copy S0 - reached through distributed shared
// memory - holds the merged tables and every decision.
struct Grp
{
	int tid, gtid, GT;        // thread in its CTA (lane for warps), thread in the group, threads in the group
	uint32_t rank, nct;       // CTA rank in the cluster, cluster size
	GroupSmem* S; GroupSmem* S0;
	uint32_t* job;            // 3 * HQ_MLP * G words of this CTA's (warp's) shared memory: clip jobs of one item tile (spatial binning)
};
template <int G> __device__ __forceinline__ void lsync() { if (G == 32) __syncwarp(); else __syncthreads(); }
template <int G> __device__ __forceinline__ void gsync( const Grp& g )
{
	if (G == 32) __syncwarp(); else if (g.nct == 1) __syncthreads(); else cg::this_cluster().sync();
}

// exclusive scan of v over the threads of the group; every thread gets the group total.  Callers pack two 16-bit
// counters into v (a tile holds at most 4096 of each).
template <int G> __device__ __forceinline__ uint32_t lscan( const Grp& g, const uint32_t v, uint32_t& total )
{
	const int lane = g.tid & 31;
	uint32_t x = v;
	#pragma unroll
	for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync( 0xffffffffu, x, o ); if (lane >= o) x += y; }
	if (G == 32) { total = __shfl_sync( 0xffffffffu, x, 31 ); return x - v; }
	GroupSmem& S = *g.S;
	const int w = g.tid >> 5;
	if (lane == 31) S.wtot[w] = x;
	__syncthreads();
	uint32_t base = 0, tot = 0;
	#pragma unroll
	for (int i = 0; i < G / 32; i++) { const uint32_t t = S.wtot[i]; if (i < w) base += t; tot += t; }
	__syncthreads();
	total = tot;
	return base + x - v;
}
template <int G> __device__ __forceinline__ uint32_t gscan( const Grp& g, const uint32_t v, uint32_t& total )
{
	uint32_t tot, base = lscan<G>( g, v, tot );
	if (G != 32 && g.nct > 1)
	{
		if (g.tid == 0) g.S0->ctot[g.rank] = tot;
		cg::this_cluster().sync();
		uint32_t cb = 0, ct = 0;
		for (uint32_t r = 0; r < g.nct; r++) { const uint32_t t = g.S0->ctot[r]; if (r < g.rank) cb += t; ct += t; }
		cg::this_cluster().sync();
		base += cb, tot = ct;
	}
	total = tot;
	return base;
}

__device__ __forceinline__ void bins_reset( GroupSmem& S, const int tid, const int G )
{
	for (int k = tid; k < 3 * HQBINS * 3; k += G) (&S.kmin[0][0][0])[k] = f2key( BVH_FAR ), (&S.kmax[0][0][0])[k] = f2key( -BVH_FAR );
	for (int k = tid; k < 3 * HQBINS; k += G) (&S.cntA[0][0])[k] = 0, (&S.cntB[0][0])[k] = 0;
}
// cluster: fold this CTA's tables into the leader's (distributed shared memory atomics)
template <int G> __device__ __forceinline__ void bins_merge( const Grp& g )
{
	if (G == 32 || g.nct == 1) return;
	__syncthreads();
	if (g.rank != 0)
	{
		GroupSmem& S = *g.S; GroupSmem& D = *g.S0;
		for (int k = g.tid; k < 3 * HQBINS * 3; k += G)
			atomicMin( &(&D.kmin[0][0][0])[k], (&S.kmin[0][0][0])[k] ), atomicMax( &(&D.kmax[0][0][0])[k], (&S.kmax[0][0][0])[k] );
		for (int k = g.tid; k < 3 * HQBINS; k += G)
			atomicAdd( &(&D.cntA[0][0])[k], (&S.cntA[0][0])[k] ), atomicAdd( &(&D.cntB[0][0])[k], (&S.cntB[0][0])[k] );
	}
}
// Shared atomics are the scarce resource of the binning loops (8192 of them per 256-thread trip), and after the first few
// fragments of a bin almost none of them changes anything: look first (a stale value only errs towards doing the atomic).
__device__ __forceinline__ void bin_grow( GroupSmem& S, const uint32_t a, const uint32_t b, const float* mn, const float* mx )
{
	#pragma unroll
	for (int k = 0; k < 3; k++)
	{
		const uint32_t lo = f2key( mn[k] ), hi = f2key( mx[k] );
		if (lo < *(volatile uint32_t*)&S.kmin[a][b][k]) atomicMin( &S.kmin[a][b][k], lo );
		if (hi > *(volatile uint32_t*)&S.kmax[a][b][k]) atomicMax( &S.kmax[a][b][k], hi );
	}
}

// One warp (all 32 lanes): the 21 candidate planes (a, i) of a node from its bin tables - prefix / suffix unions, areas,
// counts, SAH cost on lanes 0..20 - and the choice among them.
//   object split  (:2779-2803, countL = countR = cntA): first candidate in (axis, plane) order with C < splitCost, splitCost
//                 starting at noSplitCost and lowered by every accepted candidate = the first strict minimum below it;
//   spatial split (:2847-2870, countIn / countOut): the same among candidates with NL + NR < budget, NL * NR > 0 and
//                 C < 0.985 * splitCost.
// The winner lane stores the child boxes in S.best.  Returns the candidate index (-1: none) and its cost, on every lane.
__device__ __noinline__ int sweep_select( GroupSmem& S, const bool spatial, const float rSAV, const float c_trav, const float c_int,
	const bool ok0, const bool ok1, const bool ok2, const float limit, const int budget, float& bestCost, int& bestNL, int& bestNR )
{
	// lane = axis * 8 + bin: each lane decodes its own bin, then segmented (width 8) prefix and suffix unions by shuffles;
	// candidate plane i of axis a sits on lane a * 8 + i (i < 7): left = prefix of that lane, right = suffix of the next lane.
	// Lane order is candidate order.
	const int lane = (int)(threadIdx.x & 31);
	const uint32_t a = lane < 24 ? lane >> 3 : 0, i = lane & 7;
	float l1[3], l2[3], r1[3], r2[3];
	#pragma unroll
	for (int k = 0; k < 3; k++) l1[k] = r1[k] = key2f( S.kmin[a][i][k] ), l2[k] = r2[k] = key2f( S.kmax[a][i][k] );
	uint32_t lN = S.cntA[a][i], rN = spatial ? S.cntB[a][i] : lN;
	#pragma unroll
	for (int d = 1; d < 8; d <<= 1)
	{
		const bool up = (int)i >= d, dn = (int)i + d < 8;
		#pragma unroll
		for (int k = 0; k < 3; k++)
		{
			const float a1 = __shfl_up_sync( 0xffffffffu, l1[k], d, 8 ), a2 = __shfl_up_sync( 0xffffffffu, l2[k], d, 8 );
			const float b1 = __shfl_down_sync( 0xffffffffu, r1[k], d, 8 ), b2 = __shfl_down_sync( 0xffffffffu, r2[k], d, 8 );
			if (up) l1[k] = tmin( l1[k], a1 ), l2[k] = tmax( l2[k], a2 );
			if (dn) r1[k] = tmin( r1[k], b1 ), r2[k] = tmax( r2[k], b2 );
		}
		const uint32_t an = __shfl_up_sync( 0xffffffffu, lN, d, 8 ), bn = __shfl_down_sync( 0xffffffffu, rN, d, 8 );
		if (up) lN += an;
		if (dn) rN += bn;
	}
	// right side of plane i = suffix starting at bin i + 1
	#pragma unroll
	for (int k = 0; k < 3; k++) r1[k] = __shfl_down_sync( 0xffffffffu, r1[k], 1, 8 ), r2[k] = __shfl_down_sync( 0xffffffffu, r2[k], 1, 8 );
	rN = __shfl_down_sync( 0xffffffffu, rN, 1, 8 );
	const float AL = lN == 0 ? BVH_FAR : half_area3( __fsub_rn( l2[0], l1[0] ), __fsub_rn( l2[1], l1[1] ), __fsub_rn( l2[2], l1[2] ) );
	const float AR = rN == 0 ? BVH_FAR : half_area3( __fsub_rn( r2[0], r1[0] ), __fsub_rn( r2[1], r1[1] ), __fsub_rn( r2[2], r1[2] ) );
	const float C = split_cost( c_trav, c_int, rSAV, AL, (int)lN, AR, (int)rN );
	const int c = lane; // candidate id in lane space; converted to axis * 7 + plane on return
	const bool cand = lane < 24 && i < 7 && (a == 0 ? ok0 : a == 1 ? ok1 : ok2);
	int best = -1;
	if (spatial)
	{
		// NL * NR > 0 is a wrapping 32-bit product in the reference build (imul).  C < NaN and NaN < limit are both false, as in the loop.
		const bool el = cand && C < limit && (int)(lN + rN) < budget && (int)(lN * rN) > 0;
		const uint32_t m = __reduce_min_sync( 0xffffffffu, el ? f2key( C ) : 0xffffffffu );
		const uint32_t win = __ballot_sync( 0xffffffffu, el && f2key( C ) == m );
		if (win) best = __ffs( win ) - 1;
	}
	else if (__ballot_sync( 0xffffffffu, cand && C != C ) || limit != limit)
	{
		// a NaN cost (0 * inf on degenerate boxes) is "not >= splitCost" and so accepted by the reference's loop, and poisons every
		// later comparison: replay the loop literally
		float sc = limit;
		for (int k = 0; k < 24; k++)
		{
			const float Ck = __shfl_sync( 0xffffffffu, C, k );
			const bool ck = __shfl_sync( 0xffffffffu, (int)cand, k ) != 0;
			if (!ck || Ck >= sc) continue;
			sc = Ck, best = k;
		}
	}
	else
	{
		const bool el = cand && C < limit;
		const uint32_t m = __reduce_min_sync( 0xffffffffu, el ? f2key( C ) : 0xffffffffu );
		const uint32_t win = __ballot_sync( 0xffffffffu, el && f2key( C ) == m );
		if (win) best = __ffs( win ) - 1;
	}
	if (best >= 0)
	{
		if (c == best)
		{
			#pragma unroll
			for (int k = 0; k < 3; k++) S.best[k] = l1[k], S.best[3 + k] = l2[k], S.best[6 + k] = r1[k], S.best[9 + k] = r2[k];
		}
		bestCost = __shfl_sync( 0xffffffffu, C, best );
		bestNL = (int)__shfl_sync( 0xffffffffu, lN, best ), bestNR = (int)__shfl_sync( 0xffffffffu, rN, best );
		__syncwarp();
		best = (best >> 3) * 7 + (best & 7);
	}
	return best;
}

// One node, start to finish, by a group of G threads (G = 32: a warp, G = 256: a CTA).  Returns true and the two child
// tasks when the node was split.
template <int G> __device__ bool hq_node( const HQArgs& A, const Grp& g, const HQTask t, HQTask& outL, HQTask& outR )
{
	GroupSmem& S = *g.S;            // this CTA's (warp's) tables
	GroupSmem& S0 = *g.S0;          // the leader's: merged tables, decisions
	const int tid = g.tid, gtid = g.gtid, GT = g.GT;
	const bool lead = g.rank == 0;
	// TBVH_HQ_PROFILE=1: cycles of the leader thread per phase, summed over nodes (the host prints them)
	const bool prof = A.profile && lead && tid == 0;
	unsigned long long pt0 = prof ? clock64() : 0;
	#define PH( k ) do { if (prof) { const unsigned long long t1_ = clock64(); atomicAdd( &A.ctr->prof[(G == 32 ? 16 : 0) + (k)], t1_ - pt0 ); pt0 = t1_; } } while (0)
	const float4 n0 = A.tmp_nodes[(size_t)t.node * 2], n1 = A.tmp_nodes[(size_t)t.node * 2 + 1];
	const float nmin3[3] = { n0.x, n0.y, n0.z }, nmax3[3] = { n1.x, n1.y, n1.z };
	const uint32_t leftFirst = __float_as_uint( n0.w ), count = __float_as_uint( n1.w );
	const float minDim[3] = { A.ctr->min_dim[0], A.ctr->min_dim[1], A.ctr->min_dim[2] };
	const float ext[3] = { __fsub_rn( nmax3[0], nmin3[0] ), __fsub_rn( nmax3[1], nmin3[1] ), __fsub_rn( nmax3[2], nmin3[2] ) };
	const bool axisOK[3] = { ext[0] > minDim[0], ext[1] > minDim[1], ext[2] > minDim[2] };
	const float rpd3[3] = { __fdiv_rn( (float)HQBINS, ext[0] ), __fdiv_rn( (float)HQBINS, ext[1] ), __fdiv_rn( (float)HQBINS, ext[2] ) };
	const float rSAV = __fdiv_rn( 1.0f, __fmaf_rn( ext[2], ext[0], __fmaf_rn( ext[1], ext[0], __fmul_rn( ext[1], ext[2] ) ) ) );
	const float noSplitCost = __fmul_rn( __uint2float_rn( count ), A.c_int );
	const int budget = (int)(t.sliceEnd - t.sliceStart);
	const uint32_t* primIdx = A.prim_idx;

	// ---- object split: bins :2758-2775
	bins_reset( S, tid, G );
	gsync<G>( g );
	// HQ_MLP fragments per thread and trip: the index -> fragment loads of a trip are issued together
	for (uint32_t i0 = gtid; i0 < count; i0 += GT * HQ_MLP)
	{
		uint32_t fi[HQ_MLP];
		float4 fa[HQ_MLP], fb[HQ_MLP];
		#pragma unroll
		for (int u = 0; u < HQ_MLP; u++) { const uint32_t i = i0 + u * GT; fi[u] = i < count ? primIdx[leftFirst + i] : 0xffffffffu; }
		#pragma unroll
		for (int u = 0; u < HQ_MLP; u++) if (fi[u] != 0xffffffffu) fa[u] = A.frag_min[fi[u]], fb[u] = A.frag_max[fi[u]];
		#pragma unroll
		for (int u = 0; u < HQ_MLP; u++) if (fi[u] != 0xffffffffu)
		{
			const float mn[3] = { fa[u].x, fa[u].y, fa[u].z }, mx[3] = { fb[u].x, fb[u].y, fb[u].z };
			#pragma unroll
			for (int a = 0; a < 3; a++)
			{
				const int bi = clampi( cvtt( __fmul_rn( __fmaf_rn( __fadd_rn( mn[a], mx[a] ), 0.5f, -nmin3[a] ), rpd3[a] ) ), 0, HQBINS - 1 );
				bin_grow( S, a, bi, mn, mx );
				atomicAdd( &S.cntA[a][bi], 1u );
			}
		}
	}
	bins_merge<G>( g );
	gsync<G>( g );
	PH( 0 );
	if (lead && tid < 32)
	{
		float splitCost = noSplitCost;
		int nl = 0, nr = 0;
		const int best = sweep_select( S, false, rSAV, A.c_trav, A.c_int, axisOK[0], axisOK[1], axisOK[2], noSplitCost, budget, splitCost, nl, nr );
		if (tid == 0)
		{
			S.hasObj = best >= 0, S.spatial = 0, S.bestNL = S.bestNR = 0;
			bool trySpatial = false;
			if (best >= 0)
			{
				S.bestAxis = best / 7, S.bestPos = best % 7, S.bestIdx = best;
				// spatialOverlap :2806-2807: half area of (bestLMax - bestRMin) over the root's
				const float ov = __fdiv_rn( half_area3( __fsub_rn( S.best[3], S.best[6] ), __fsub_rn( S.best[4], S.best[7] ), __fsub_rn( S.best[5], S.best[8] ) ), A.ctr->root_area );
				trySpatial = ov > 1e-4f;
			}
			// without an object candidate splitCost == noSplitCost and the reference's second disjunct holds whatever its stale bounds say
			trySpatial = (budget > (int)count) && (trySpatial || splitCost >= noSplitCost);
			S.splitCost = splitCost, S.trySpatial = trySpatial;
		}
	}
	gsync<G>( g );
	PH( 1 );

	// ---- spatial split candidate :2808-2872
	if (S0.trySpatial)
	{
		bins_reset( S, tid, G );
		gsync<G>( g );
		const float planeDist3[3] = { __fdiv_rn( ext[0], __fmul_rn( (float)HQBINS, 0.9999f ) ), __fdiv_rn( ext[1], __fmul_rn( (float)HQBINS, 0.9999f ) ), __fdiv_rn( ext[2], __fmul_rn( (float)HQBINS, 0.9999f ) ) };
		// items are (fragment, axis) pairs; an item that spans several bins becomes one clip job per bin (:2831-2845).  The
		// jobs of a tile of items are spread over all threads of the CTA (warp), whichever thread owned the item.
		// kpp items per thread and tile (HQ_MLP for big nodes, 1 when the node has no more items than the group has threads)
		const uint32_t items = count * 3, kpp = min( (uint32_t)HQ_MLP, (items + (uint32_t)GT - 1) / (uint32_t)GT );
		uint32_t* job_off = g.job, * job_fi = g.job + HQ_MLP * G, * job_ab = g.job + 2 * HQ_MLP * G;
		for (uint32_t base = 0; base < items; base += GT * kpp)
		{
			uint32_t nb[HQ_MLP], fi[HQ_MLP], ab[HQ_MLP], nbsum = 0;
			float4 fa[HQ_MLP], fb[HQ_MLP];
			#pragma unroll
			for (int u = 0; u < HQ_MLP; u++)
			{
				const uint32_t it = base + gtid * kpp + u, i = it / 3, a = it - i * 3;
				nb[u] = 0, ab[u] = a, fi[u] = 0xffffffffu;
				if (u < (int)kpp && it < items && (a == 0 ? axisOK[0] : a == 1 ? axisOK[1] : axisOK[2])) fi[u] = primIdx[leftFirst + i];
			}
			#pragma unroll
			for (int u = 0; u < HQ_MLP; u++) if (fi[u] != 0xffffffffu) fa[u] = A.frag_min[fi[u]], fb[u] = A.frag_max[fi[u]];
			#pragma unroll
			for (int u = 0; u < HQ_MLP; u++) if (fi[u] != 0xffffffffu)
			{
				const uint32_t a = ab[u];
				const float planeDist = a == 0 ? planeDist3[0] : a == 1 ? planeDist3[1] : planeDist3[2];
				const float rPlaneDist = __fdiv_rn( 1.0f, planeDist ), nodeMin = a == 0 ? nmin3[0] : a == 1 ? nmin3[1] : nmin3[2];
				const int bin1 = clampi( cvtt( __fmul_rn( __fsub_rn( comp( fa[u], a ), nodeMin ), rPlaneDist ) ), 0, HQBINS - 1 );
				const int bin2 = clampi( cvtt( __fmul_rn( __fsub_rn( comp( fb[u], a ), nodeMin ), rPlaneDist ) ), 0, HQBINS - 1 );
				atomicAdd( &S.cntA[a][bin1], 1u ), atomicAdd( &S.cntB[a][bin2], 1u );
				if (bin2 == bin1)
				{
					const float mn[3] = { fa[u].x, fa[u].y, fa[u].z }, mx[3] = { fb[u].x, fb[u].y, fb[u].z };
					bin_grow( S, a, bin1, mn, mx );
				}
				else nb[u] = (uint32_t)(bin2 - bin1 + 1), ab[u] = a | ((uint32_t)bin1 << 2);
				nbsum += nb[u];
			}
			uint32_t T, off = lscan<G>( g, nbsum, T );
			if (T == 0) continue; // uniform within the CTA (warp)
			#pragma unroll
			for (int u = 0; u < HQ_MLP; u++)
			{
				const uint32_t e = (uint32_t)tid * HQ_MLP + u;
				job_off[e] = off, job_fi[e] = fi[u], job_ab[e] = ab[u];
				off += nb[u];
			}
			lsync<G>();
			for (uint32_t q = tid; q < T; q += G)
			{
				// owner = last item whose first job is <= q (items without jobs share their successor's offset and are skipped by this)
				uint32_t lo = 0, hi = G * HQ_MLP;
				while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (job_off[mid] <= q) lo = mid; else hi = mid; }
				const uint32_t a = job_ab[lo] & 3u;
				const int j = (int)(job_ab[lo] >> 2) + (int)(q - job_off[lo]);
				const Frag f = load_frag( A, job_fi[lo] );
				const float planeDist = a == 0 ? planeDist3[0] : a == 1 ? planeDist3[1] : planeDist3[2];
				float bmin[3] = { nmin3[0], nmin3[1], nmin3[2] }, bmax[3] = { nmax3[0], nmax3[1], nmax3[2] }, nbmin[3], nbmax[3];
				const float lo_a = __fmaf_rn( __int2float_rn( j ), planeDist, a == 0 ? nmin3[0] : a == 1 ? nmin3[1] : nmin3[2] );
				const float hi_a = j == HQBINS - 2 ? (a == 0 ? nmax3[0] : a == 1 ? nmax3[1] : nmax3[2]) : __fadd_rn( lo_a, planeDist );
				if (a == 0) bmin[0] = lo_a, bmax[0] = hi_a; else if (a == 1) bmin[1] = lo_a, bmax[1] = hi_a; else bmin[2] = lo_a, bmax[2] = hi_a;
				if (!clip_frag( A, f, nbmin, nbmax, bmin, bmax, minDim, a )) continue;
				bin_grow( S, a, (uint32_t)j, nbmin, nbmax );
			}
			lsync<G>();
		}
		bins_merge<G>( g );
		gsync<G>( g );
		PH( 2 );
		if (lead && tid < 32)
		{
			float splitCost = S.splitCost;
			int nl = 0, nr = 0;
			const int best = sweep_select( S, true, rSAV, A.c_trav, A.c_int, axisOK[0], axisOK[1], axisOK[2], __fmul_rn( splitCost, 0.985f ), budget, splitCost, nl, nr );
			if (best >= 0 && tid == 0)
			{
				const uint32_t a = best / 7;
				S.spatial = 1, S.bestAxis = a, S.bestPos = best % 7, S.bestIdx = best, S.splitCost = splitCost;
				S.bestNL = nl, S.bestNR = nr;
				S.best[3 + a] = S.best[6 + a]; // bestLMax[a] = bestRMin[a], "accurate" :2868
			}
		}
		gsync<G>( g );
		PH( 3 );
	}

	// ---- leaf? :2874-2880
	if (S0.splitCost >= noSplitCost)
	{
		for (uint32_t i = gtid; i < count; i += GT) { const uint32_t p = leftFirst + i; A.prim_idx[p] = __float_as_uint( A.frag_min[A.prim_idx[p]].w ); }
		if (lead && tid == 0) atomicMax( &A.ctr->max_depth, t.depth );
		gsync<G>( g ); // nobody reads the leader's tables after it has moved on
		PH( 9 );
		return false;
	}

	// ---- partition into idxTmp :2882-2964
	const uint32_t bestAxis = S0.bestAxis, bestPos = S0.bestPos;
	const bool spatial = S0.spatial != 0;
	uint32_t Apos = t.sliceStart, Bpos = t.sliceEnd;
	// consecutive fragments per thread in the scan tiles of the partition passes: HQ_E for big nodes (fewer group-wide scans),
	// down to 1 when the node has no more fragments than the group has threads
	const uint32_t epp = min( (uint32_t)HQ_E, (count + (uint32_t)GT - 1) / (uint32_t)GT );
	if (!spatial)
	{
		const float rpd = rpd3[bestAxis], nmin = nmin3[bestAxis];
		for (uint32_t base = 0; base < count; base += GT * epp)
		{
			uint32_t fr[HQ_E], flag[HQ_E], sum = 0;
			#pragma unroll
			for (int e = 0; e < HQ_E; e++)
			{
				const uint32_t i = base + gtid * epp + e;
				fr[e] = flag[e] = 0;
				if (e < (int)epp && i < count)
				{
					fr[e] = primIdx[leftFirst + i];
					const float mn = comp( A.frag_min[fr[e]], bestAxis ), mx = comp( A.frag_max[fr[e]], bestAxis );
					const int bi = clampi( cvtt( __fmul_rn( __fmaf_rn( __fadd_rn( mn, mx ), 0.5f, -nmin ), rpd ) ), 0, HQBINS - 1 );
					flag[e] = bi <= (int)bestPos ? 1u : 0x10000u;
				}
				sum += flag[e];
			}
			uint32_t tot, run = gscan<G>( g, sum, tot );
			#pragma unroll
			for (int e = 0; e < HQ_E; e++)
			{
				if (flag[e] == 1u) A.idx_tmp[Apos + (run & 0xffffu)] = fr[e];
				else if (flag[e]) A.idx_tmp[Bpos - 1 - (run >> 16)] = fr[e];
				run += flag[e];
			}
			Apos += tot & 0xffffu, Bpos -= tot >> 16;
		}
		PH( 4 );
	}
	else
	{
		const float planeDist = __fdiv_rn( ext[bestAxis], __fmul_rn( (float)HQBINS, 0.9999f ) );
		const float rPlaneDist = __fdiv_rn( 1.0f, planeDist ), nodeMin = nmin3[bestAxis];
		uint32_t* cls = A.cls + t.sliceStart, * strad = A.strad + t.sliceStart;
		float* spos = A.spos + t.sliceStart;
		// pass 1: left / right / straddler, straddlers listed in order
		uint32_t nstrad = 0;
		for (uint32_t base = 0; base < count; base += GT * epp)
		{
			uint32_t flags = 0;
			#pragma unroll
			for (int e = 0; e < HQ_E; e++)
			{
				const uint32_t i = base + gtid * epp + e;
				if (e < (int)epp && i < count)
				{
					const uint32_t fr = primIdx[leftFirst + i];
					const float mn = comp( A.frag_min[fr], bestAxis ), mx = comp( A.frag_max[fr], bestAxis );
					const uint32_t bin1 = __float2uint_rz( tmax( __fmul_rn( __fsub_rn( mn, nodeMin ), rPlaneDist ), 0.0f ) );
					const uint32_t bin2 = __float2uint_rz( tmax( __fmul_rn( __fsub_rn( mx, nodeMin ), rPlaneDist ), 0.0f ) );
					const uint32_t c = bin2 <= bestPos ? 0u : bin1 > bestPos ? 1u : 2u;
					cls[i] = c;
					if (c == 2u) flags |= 1u << e;
				}
			}
			uint32_t tot, run = gscan<G>( g, (uint32_t)__popc( flags ), tot );
			#pragma unroll
			for (int e = 0; e < HQ_E; e++) if (flags & (1u << e)) strad[nstrad + run++] = base + gtid * epp + e;
			nstrad += tot;
		}
		gsync<G>( g );
		PH( 5 );
		// pass 2: the unsplitting chain :2895-2926, one warp, in order.  A straddler that ends up split leaves the running
		// state (child boxes, counts, cost) untouched, and most do: the 32 straddlers of a batch are judged in parallel
		// against the current state, everything up to the first one that unsplits is final, that one commits and
		// broadcasts its new state, the lanes behind it are judged again.
		if (lead && tid < 32)
		{
			int NL = S.bestNL, NR = S.bestNR;
			float cost = S.splitCost, LMin[3], LMax[3], RMin[3], RMax[3];
			#pragma unroll
			for (int k = 0; k < 3; k++) LMin[k] = S.best[k], LMax[k] = S.best[3 + k], RMin[k] = S.best[6 + k], RMax[k] = S.best[9 + k];
			for (uint32_t base = 0; base < nstrad; base += 32)
			{
				const uint32_t k = base + tid;
				const bool valid = k < nstrad;
				float4 fa = make_float4( 0, 0, 0, 0 ), fb = fa;
				uint32_t i = 0;
				if (valid) { i = strad[k]; const uint32_t fr = primIdx[leftFirst + i]; fa = A.frag_min[fr], fb = A.frag_max[fr]; }
				const float fmn[3] = { fa.x, fa.y, fa.z }, fmx[3] = { fb.x, fb.y, fb.z };
				uint32_t mydec = 2, start = 0;
				float mypos = 0;
				for (;;)
				{
					uint32_t dec = 2;
					float uMin[3], uMax[3], C = 0;
					if (valid && (uint32_t)tid >= start)
					{
						if (NR > 1)
						{
							#pragma unroll
							for (int q = 0; q < 3; q++) uMin[q] = tmin( LMin[q], fmn[q] ), uMax[q] = tmax( LMax[q], fmx[q] );
							const float AL = half_area3( __fsub_rn( uMax[0], uMin[0] ), __fsub_rn( uMax[1], uMin[1] ), __fsub_rn( uMax[2], uMin[2] ) );
							const float AR = half_area3( __fsub_rn( RMax[0], RMin[0] ), __fsub_rn( RMax[1], RMin[1] ), __fsub_rn( RMax[2], RMin[2] ) );
							C = split_cost( A.c_trav, A.c_int, rSAV, AL, NL, AR, NR - 1 );
							if (C <= cost) dec = 0;
						}
						if (dec == 2 && NL > 1)
						{
							#pragma unroll
							for (int q = 0; q < 3; q++) uMin[q] = tmin( RMin[q], fmn[q] ), uMax[q] = tmax( RMax[q], fmx[q] );
							const float AL = half_area3( __fsub_rn( LMax[0], LMin[0] ), __fsub_rn( LMax[1], LMin[1] ), __fsub_rn( LMax[2], LMin[2] ) );
							const float AR = half_area3( __fsub_rn( uMax[0], uMin[0] ), __fsub_rn( uMax[1], uMin[1] ), __fsub_rn( uMax[2], uMin[2] ) );
							C = split_cost( A.c_trav, A.c_int, rSAV, AL, NL - 1, AR, NR );
							if (C <= cost) dec = 1;
						}
					}
					const uint32_t changed = __ballot_sync( 0xffffffffu, dec != 2 );
					const uint32_t first = changed ? (uint32_t)__ffs( changed ) - 1u : 32u;
					if ((uint32_t)tid >= start && (uint32_t)tid < first) mydec = 2, mypos = bestAxis == 0 ? LMax[0] : bestAxis == 1 ? LMax[1] : LMax[2];
					if (first == 32u) break;
					if ((uint32_t)tid == first) mydec = dec;
					const uint32_t d = __shfl_sync( 0xffffffffu, dec, first );
					cost = __shfl_sync( 0xffffffffu, C, first );
					float bMin[3], bMax[3];
					#pragma unroll
					for (int q = 0; q < 3; q++) bMin[q] = __shfl_sync( 0xffffffffu, uMin[q], first ), bMax[q] = __shfl_sync( 0xffffffffu, uMax[q], first );
					if (d == 0)
					{
						NR--;
						#pragma unroll
						for (int q = 0; q < 3; q++) LMin[q] = bMin[q], LMax[q] = bMax[q];
					}
					else
					{
						NL--;
						#pragma unroll
						for (int q = 0; q < 3; q++) RMin[q] = bMin[q], RMax[q] = bMax[q];
					}
					start = first + 1;
				}
				if (valid) cls[i] = mydec, spos[k] = mypos;
			}
		}
		gsync<G>( g );
		PH( 6 );
		// pass 3: clip the fragments the chain decided to split :2927-2941
		for (uint32_t k = gtid; k < nstrad; k += GT)
		{
			const uint32_t i = strad[k];
			if (cls[i] != 2u) continue;
			const uint32_t fragIdx = primIdx[leftFirst + i];
			const Frag f = load_frag( A, fragIdx );
			float lmin[3], lmax[3], rmin[3], rmax[3];
			bool leftOK, rightOK;
			split_frag( A, f, lmin, lmax, rmin, rmax, minDim, bestAxis, spos[k], leftOK, rightOK );
			if (leftOK && rightOK)
			{
				const uint32_t nf = atomicAdd( &A.ctr->frag_ptr, 1u );
				if (nf >= A.idx_cap) { atomicAdd( &A.ctr->overflow, 1u ); cls[i] = 0u; continue; }
				store_frag( A, fragIdx, lmin, lmax, f.prim ), store_frag( A, nf, rmin, rmax, f.prim );
				cls[i] = 0x80000000u | nf;
			}
			else cls[i] = leftOK ? 0u : 1u;
		}
		gsync<G>( g );
		PH( 7 );
		// pass 4: left part upward from sliceStart, right part downward from sliceEnd, in fragment order
		for (uint32_t base = 0; base < count; base += GT * epp)
		{
			uint32_t fr[HQ_E], c[HQ_E], flag[HQ_E], sum = 0;
			#pragma unroll
			for (int e = 0; e < HQ_E; e++)
			{
				const uint32_t i = base + gtid * epp + e;
				fr[e] = c[e] = flag[e] = 0;
				if (e < (int)epp && i < count)
				{
					fr[e] = primIdx[leftFirst + i], c[e] = cls[i];
					flag[e] = (c[e] & 0x80000000u) ? 0x10001u : c[e] == 0u ? 1u : 0x10000u;
				}
				sum += flag[e];
			}
			uint32_t tot, run = gscan<G>( g, sum, tot );
			#pragma unroll
			for (int e = 0; e < HQ_E; e++)
			{
				if (flag[e] & 1u) A.idx_tmp[Apos + (run & 0xffffu)] = fr[e];
				if (flag[e] >> 16) A.idx_tmp[Bpos - 1 - (run >> 16)] = (c[e] & 0x80000000u) ? (c[e] & 0x7fffffffu) : fr[e];
				run += flag[e];
			}
			Apos += tot & 0xffffu, Bpos -= tot >> 16;
		}
		// child bounds are refreshed from the fragments :2943-2950
		for (int k = tid; k < 12; k += G) S.ckey[k] = ((k / 3) & 1) ? f2key( -BVH_FAR ) : f2key( BVH_FAR );
		gsync<G>( g );
		const uint32_t nl = Apos - t.sliceStart, nr = t.sliceEnd - Bpos;
		{
			// per-thread boxes over its fragments, one redux per word and warp, one shared atomic per word and warp
			uint32_t bk[12];
			#pragma unroll
			for (int k = 0; k < 12; k++) bk[k] = ((k / 3) & 1) ? f2key( -BVH_FAR ) : f2key( BVH_FAR );
			for (uint32_t base = 0; base < nl + nr; base += GT * HQ_MLP)
			{
				uint32_t fr[HQ_MLP];
				#pragma unroll
				for (int u = 0; u < HQ_MLP; u++)
				{
					const uint32_t i = base + gtid + u * GT;
					fr[u] = i < nl + nr ? A.idx_tmp[i >= nl ? Bpos + (i - nl) : t.sliceStart + i] : 0xffffffffu;
				}
				#pragma unroll
				for (int u = 0; u < HQ_MLP; u++) if (fr[u] != 0xffffffffu)
				{
					const float4 fa = A.frag_min[fr[u]], fb = A.frag_max[fr[u]];
					const uint32_t ka[6] = { f2key( fa.x ), f2key( fa.y ), f2key( fa.z ), f2key( fb.x ), f2key( fb.y ), f2key( fb.z ) };
					if (base + gtid + u * GT >= nl)
					{
						#pragma unroll
						for (int q = 0; q < 3; q++) bk[6 + q] = min( bk[6 + q], ka[q] ), bk[9 + q] = max( bk[9 + q], ka[3 + q] );
					}
					else
					{
						#pragma unroll
						for (int q = 0; q < 3; q++) bk[q] = min( bk[q], ka[q] ), bk[3 + q] = max( bk[3 + q], ka[3 + q] );
					}
				}
			}
			__syncwarp();
			#pragma unroll
			for (int k = 0; k < 12; k++)
			{
				const uint32_t r = ((k / 3) & 1) ? __reduce_max_sync( 0xffffffffu, bk[k] ) : __reduce_min_sync( 0xffffffffu, bk[k] );
				if ((tid & 31) == 0) { if ((k / 3) & 1) atomicMax( &S.ckey[k], r ); else atomicMin( &S.ckey[k], r ); }
			}
		}
		if (G != 32 && g.nct > 1)
		{
			__syncthreads();
			if (!lead && tid < 12) { if ((tid / 3) & 1) atomicMax( &S0.ckey[tid], S.ckey[tid] ); else atomicMin( &S0.ckey[tid], S.ckey[tid] ); }
		}
		gsync<G>( g );
		if (lead && tid < 12) S.best[tid] = key2f( S.ckey[tid] );
		PH( 8 );
	}
	gsync<G>( g );
	// copy back :2965 (the parts that hold fragments; the rest of the slice is never read through primIdx)
	const uint32_t leftCount = Apos - t.sliceStart, rightCount = t.sliceEnd - Bpos;
	for (uint32_t i = gtid; i < leftCount + rightCount; i += GT)
	{
		const uint32_t p = i < leftCount ? t.sliceStart + i : Bpos + (i - leftCount);
		A.prim_idx[p] = A.idx_tmp[p];
	}
	gsync<G>( g );
	PH( 10 );
	if (leftCount == 0 || rightCount == 0)
	{
		// ":2939 spatial split failed": the reference reads the node's OLD range out of the refreshed primIdx, i.e. whatever
		// idxTmp holds there (this node's own output where the ranges overlap, an ancestor's words or zeros elsewhere)
		for (uint32_t i = gtid; i < count; i += GT) { const uint32_t p = leftFirst + i; A.prim_idx[p] = __float_as_uint( A.frag_min[A.idx_tmp[p]].w ); }
		if (lead && tid == 0)
		{
			const float* b = S.best;
			A.tmp_nodes[(size_t)t.node * 2] = make_float4( tmin( b[0], b[6] ), tmin( b[1], b[7] ), tmin( b[2], b[8] ), n0.w );
			A.tmp_nodes[(size_t)t.node * 2 + 1] = make_float4( tmax( b[3], b[9] ), tmax( b[4], b[10] ), tmax( b[5], b[11] ), n1.w );
			atomicAdd( &A.ctr->failed_splits, 1u ), atomicMax( &A.ctr->max_depth, t.depth );
		}
		gsync<G>( g );
		return false;
	}
	// ---- emit :2966-2984
	if (lead && tid == 0)
	{
		const uint32_t lc = atomicAdd( &A.ctr->node_ptr, 2u );
		S.lc = lc;
		if (lc + 2 <= A.node_cap)
		{
			const float* b = S.best;
			A.tmp_nodes[(size_t)lc * 2] = make_float4( b[0], b[1], b[2], __uint_as_float( t.sliceStart ) );
			A.tmp_nodes[(size_t)lc * 2 + 1] = make_float4( b[3], b[4], b[5], __uint_as_float( leftCount ) );
			A.tmp_nodes[(size_t)lc * 2 + 2] = make_float4( b[6], b[7], b[8], __uint_as_float( Bpos ) );
			A.tmp_nodes[(size_t)lc * 2 + 3] = make_float4( b[9], b[10], b[11], __uint_as_float( rightCount ) );
			A.tmp_nodes[(size_t)t.node * 2] = make_float4( n0.x, n0.y, n0.z, __uint_as_float( lc ) );
			A.tmp_nodes[(size_t)t.node * 2 + 1] = make_float4( n1.x, n1.y, n1.z, __uint_as_float( 0u ) );
			A.parent[lc] = A.parent[lc + 1] = t.node;
		}
		else atomicAdd( &A.ctr->overflow, 1u );
	}
	gsync<G>( g );
	const uint32_t lc = S0.lc;
	const uint32_t mid = (Apos + Bpos) >> 1;
	outL.node = lc, outL.sliceStart = t.sliceStart, outL.sliceEnd = mid, outL.depth = t.depth + 1;
	outR.node = lc + 1, outR.sliceStart = mid, outR.sliceEnd = t.sliceEnd, outR.depth = t.depth + 1;
	gsync<G>( g );
	PH( 11 );
	#undef PH
	return lc + 2 <= A.node_cap;
}

// ---------------------------------------------------------------------------------------------- kernels
__global__ void k_hq_init( HQArgs A )
{
	HQCounters* c = A.ctr;
	c->node_ptr = 2, c->frag_ptr = A.n, c->next_big = 0, c->small_roots = 0, c->max_depth = 0, c->next_max = 0, c->failed_splits = 0, c->overflow = 0;
	for (int k = 0; k < 3; k++) c->root_key[k] = f2key( BVH_FAR ), c->root_key[3 + k] = f2key( -BVH_FAR );
	for (int k = 0; k < 32; k++) c->prof[k] = 0;
}

// PrepareHQBuild :2677-2686: fragment boxes, identity primIdx, root bounds
__global__ void k_hq_fragments( HQArgs A )
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	float mn[3] = { BVH_FAR, BVH_FAR, BVH_FAR }, mx[3] = { -BVH_FAR, -BVH_FAR, -BVH_FAR };
	if (i < A.n)
	{
		const float4 v0 = A.verts[(size_t)i * 3], v1 = A.verts[(size_t)i * 3 + 1], v2 = A.verts[(size_t)i * 3 + 2];
		mn[0] = tmin( v0.x, tmin( v1.x, v2.x ) ), mn[1] = tmin( v0.y, tmin( v1.y, v2.y ) ), mn[2] = tmin( v0.z, tmin( v1.z, v2.z ) );
		mx[0] = tmax( v0.x, tmax( v1.x, v2.x ) ), mx[1] = tmax( v0.y, tmax( v1.y, v2.y ) ), mx[2] = tmax( v0.z, tmax( v1.z, v2.z ) );
		A.frag_min[i] = make_float4( mn[0], mn[1], mn[2], __uint_as_float( i ) );
		A.frag_max[i] = make_float4( mx[0], mx[1], mx[2], __uint_as_float( 0u ) );
		A.prim_idx[i] = i;
	}
	#pragma unroll
	for (int k = 0; k < 3; k++)
	{
		uint32_t a = f2key( mn[k] ), b = f2key( mx[k] );
		a = __reduce_min_sync( 0xffffffffu, a ), b = __reduce_max_sync( 0xffffffffu, b );
		if ((threadIdx.x & 31) == 0) atomicMin( &A.ctr->root_key[k], a ), atomicMax( &A.ctr->root_key[3 + k], b );
	}
}

__global__ void k_hq_root( HQArgs A )
{
	HQCounters* c = A.ctr;
	float mn[3], mx[3];
	for (int k = 0; k < 3; k++) mn[k] = key2f( c->root_key[k] ), mx[k] = key2f( c->root_key[3 + k] );
	A.tmp_nodes[0] = make_float4( mn[0], mn[1], mn[2], __uint_as_float( 0u ) );
	A.tmp_nodes[1] = make_float4( mx[0], mx[1], mx[2], __uint_as_float( A.n ) );
	A.tmp_nodes[2] = A.tmp_nodes[3] = make_float4( 0, 0, 0, 0 );
	A.parent[0] = A.parent[1] = 0xffffffffu;
	const float ex = __fsub_rn( mx[0], mn[0] ), ey = __fsub_rn( mx[1], mn[1] ), ez = __fsub_rn( mx[2], mn[2] );
	c->root_area = half_area3( ex, ey, ez );
	c->min_dim[0] = __fmul_rn( ex, 1e-7f ), c->min_dim[1] = __fmul_rn( ey, 1e-7f ), c->min_dim[2] = __fmul_rn( ez, 1e-7f );
	HQTask t = { 0u, 0u, A.idx_cap, 0u };
	if (A.n > HQ_SMALL) A.lvl[0][0] = t, c->next_big = 1, c->next_max = A.n; else A.small[0] = t, c->small_roots = 1;
}

__device__ __forceinline__ void hq_enqueue( const HQArgs& A, HQTask* next, const HQTask c )
{
	const uint32_t cnt = __float_as_uint( A.tmp_nodes[(size_t)c.node * 2 + 1].w );
	if (cnt > HQ_SMALL)
	{
		atomicMax( &A.ctr->next_max, cnt );
		const uint32_t k = atomicAdd( &A.ctr->next_big, 1u );
		if (k < A.lvl_cap) next[k] = c; else atomicAdd( &A.ctr->overflow, 1u );
	}
	else A.small[atomicAdd( &A.ctr->small_roots, 1u )] = c;
}

// level-synchronous phase: one cluster of nct CTAs (run-time cluster dimension, 1..16) per node
__global__ void __launch_bounds__( HQ_BIG_THREADS, 3 ) k_hq_level( HQArgs A, const HQTask* cur, HQTask* next, const uint32_t nct )
{
	__shared__ GroupSmem S;
	__shared__ uint32_t job[3 * HQ_MLP * HQ_BIG_THREADS];
	Grp g;
	g.tid = (int)threadIdx.x, g.nct = nct, g.rank = 0, g.S = g.S0 = &S, g.job = job;
	if (nct > 1)
	{
		cg::cluster_group cl = cg::this_cluster();
		g.rank = cl.block_rank(), g.S0 = cl.map_shared_rank( &S, 0 );
	}
	g.gtid = (int)(g.rank * HQ_BIG_THREADS + threadIdx.x), g.GT = (int)(nct * HQ_BIG_THREADS);
	HQTask l, r;
	const bool split = hq_node<HQ_BIG_THREADS>( A, g, cur[blockIdx.x / nct], l, r );
	if (split && g.rank == 0 && threadIdx.x == 0) hq_enqueue( A, next, l ), hq_enqueue( A, next, r );
}

__global__ void __launch_bounds__( HQ_SMALL_WARPS * 32, 6 ) k_hq_subtrees( HQArgs A, const uint32_t roots )
{
	__shared__ GroupSmem Ss[HQ_SMALL_WARPS];
	__shared__ HQTask stack[HQ_SMALL_WARPS][HQ_STACK];
	__shared__ uint32_t job[HQ_SMALL_WARPS][3 * HQ_MLP * 32];
	const uint32_t w = threadIdx.x >> 5, lane = threadIdx.x & 31, id = blockIdx.x * HQ_SMALL_WARPS + w;
	if (id >= roots) return;
	Grp g;
	g.tid = g.gtid = (int)lane, g.GT = 32, g.rank = 0, g.nct = 1, g.S = g.S0 = &Ss[w], g.job = job[w];
	HQTask t = A.small[id];
	uint32_t sp = 0;
	for (;;)
	{
		HQTask l, r;
		if (hq_node<32>( A, g, t, l, r ))
		{
			// continue with the child that holds fewer fragments, park the other: the stack stays logarithmic
			const uint32_t cl = __float_as_uint( A.tmp_nodes[(size_t)l.node * 2 + 1].w ), cr = __float_as_uint( A.tmp_nodes[(size_t)r.node * 2 + 1].w );
			const HQTask park = cl <= cr ? r : l;
			t = cl <= cr ? l : r;
			if (sp < HQ_STACK) { if (lane == 0) stack[w][sp] = park; sp++; }
			else if (lane == 0) atomicAdd( &A.ctr->overflow, 1u );
			__syncwarp();
			continue;
		}
		if (!sp) break;
		t = stack[w][--sp];
		__syncwarp();
	}
}

// ---- Compact() :3733-3770 as a parallel relayout
// bottom-up: number of interior nodes / of leaf index entries per subtree (second arrival at a parent carries on)
__global__ void k_hq_up( HQArgs A, const uint32_t tmp_count )
{
	uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
	if (x >= tmp_count || x == 1) return;
	const uint32_t cnt = __float_as_uint( A.tmp_nodes[(size_t)x * 2 + 1].w );
	if (cnt == 0) return; // interior
	A.sub_int[x] = 0, A.sub_prims[x] = cnt;
	for (;;)
	{
		const uint32_t p = A.parent[x];
		if (p == 0xffffffffu) break;
		__threadfence();
		if (atomicAdd( &A.arrive[p], 1u ) == 0) break;
		__threadfence();
		const uint32_t lc = __float_as_uint( A.tmp_nodes[(size_t)p * 2].w );
		const volatile uint32_t* si = A.sub_int; const volatile uint32_t* sp = A.sub_prims;
		A.sub_int[p] = si[lc] + si[lc + 1] + 1, A.sub_prims[p] = sp[lc] + sp[lc + 1];
		x = p;
	}
}
// top-down by walking to the root: K = interior nodes before x in DFS preorder, O = leaf index entries before x
__global__ void k_hq_down( HQArgs A, const uint32_t tmp_count, float4* out_nodes, uint32_t* out_idx )
{
	const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
	if (x >= tmp_count) return;
	if (x == 1) { out_nodes[2] = out_nodes[3] = make_float4( 0, 0, 0, 0 ); return; }
	uint32_t K = 0, O = 0, c = x, Kparent = 0;
	while (c != 0)
	{
		const uint32_t p = A.parent[c], lc = __float_as_uint( A.tmp_nodes[(size_t)p * 2].w );
		uint32_t add = 1;
		if (c == lc + 1) add += A.sub_int[lc], O += A.sub_prims[lc];
		if (c == x) Kparent = add; // K(parent) = K(x) - add, fixed up below
		K += add, c = p;
	}
	const uint32_t dst = x == 0 ? 0u : 2u + 2u * (K - Kparent) + ((x & 1u) ? 1u : 0u); // pairs start at even temp indices: odd = right child
	const float4 a = A.tmp_nodes[(size_t)x * 2], b = A.tmp_nodes[(size_t)x * 2 + 1];
	const uint32_t cnt = __float_as_uint( b.w );
	if (cnt == 0) out_nodes[(size_t)dst * 2] = make_float4( a.x, a.y, a.z, __uint_as_float( 2u + 2u * K ) ), out_nodes[(size_t)dst * 2 + 1] = b;
	else
	{
		out_nodes[(size_t)dst * 2] = make_float4( a.x, a.y, a.z, __uint_as_float( O ) ), out_nodes[(size_t)dst * 2 + 1] = b;
		const uint32_t first = __float_as_uint( a.w );
		for (uint32_t i = 0; i < cnt; i++) out_idx[O + i] = A.prim_idx[first + i];
	}
}
} // namespace

#define DEV_ALLOC( p, bytes ) do { void* q_ = 0; CUDA_TRY( cudaMalloc( &q_, (bytes) ) ); scratch.push_back( q_ ); (p) = (decltype( p ))q_; } while (0)

int build_hq_launch( tbvh_bvh b, float c_trav, float c_int )
{
	const uint32_t n = b->info.prim_count, slack = n >> 1;
	cudaStream_t s = b->ctx->stream;
	std::vector<void*> scratch;
	HQArgs A = {};
	A.verts = b->d_verts, A.n = n, A.c_trav = c_trav, A.c_int = c_int;
	A.idx_cap = n + slack, A.node_cap = 3 * n + 2;
	A.lvl_cap = A.idx_cap / HQ_SMALL + 2;
	{ const char* e = getenv( "TBVH_HQ_PROFILE" ); A.profile = e ? (uint32_t)atoi( e ) : 0u; }
	HQCounters* h_ctr = 0;
	cudaEvent_t e0 = 0, e1 = 0;
	CUDA_TRY( cudaMalloc( &b->d_nodes, (size_t)A.node_cap * 32 ) );
	CUDA_TRY( cudaMalloc( &b->d_prim_idx, (size_t)A.idx_cap * 4 ) );
	auto body = [&]() -> int
	{
		DEV_ALLOC( A.frag_min, (size_t)A.idx_cap * 16 ); DEV_ALLOC( A.frag_max, (size_t)A.idx_cap * 16 );
		DEV_ALLOC( A.prim_idx, (size_t)A.idx_cap * 4 ); DEV_ALLOC( A.idx_tmp, (size_t)A.idx_cap * 4 );
		DEV_ALLOC( A.cls, (size_t)A.idx_cap * 4 ); DEV_ALLOC( A.strad, (size_t)A.idx_cap * 4 ); DEV_ALLOC( A.spos, (size_t)A.idx_cap * 4 );
		DEV_ALLOC( A.tmp_nodes, (size_t)A.node_cap * 32 ); DEV_ALLOC( A.parent, (size_t)A.node_cap * 4 );
		DEV_ALLOC( A.sub_int, (size_t)A.node_cap * 4 ); DEV_ALLOC( A.sub_prims, (size_t)A.node_cap * 4 ); DEV_ALLOC( A.arrive, (size_t)A.node_cap * 4 );
		DEV_ALLOC( A.lvl[0], (size_t)A.lvl_cap * sizeof( HQTask ) ); DEV_ALLOC( A.lvl[1], (size_t)A.lvl_cap * sizeof( HQTask ) );
		DEV_ALLOC( A.small, ((size_t)A.idx_cap + 1) * sizeof( HQTask ) );
		DEV_ALLOC( A.ctr, sizeof( HQCounters ) );
		CUDA_TRY( cudaMallocHost( &h_ctr, sizeof( HQCounters ) ) );
		CUDA_TRY( cudaEventCreate( &e0 ) ); CUDA_TRY( cudaEventCreate( &e1 ) );
		CUDA_TRY( cudaEventRecord( e0, s ) );
		// the reference clears primIdx beyond triCount (:2700) and all of idxTmp (:3008)
		CUDA_TRY( cudaMemsetAsync( A.prim_idx, 0, (size_t)A.idx_cap * 4, s ) );
		CUDA_TRY( cudaMemsetAsync( A.idx_tmp, 0, (size_t)A.idx_cap * 4, s ) );
		CUDA_TRY( cudaMemsetAsync( A.arrive, 0, (size_t)A.node_cap * 4, s ) );
		k_hq_init<<<1, 1, 0, s>>>( A ); LAUNCHED();
		k_hq_fragments<<<(n + 255) / 256, 256, 0, s>>>( A ); LAUNCHED();
		k_hq_root<<<1, 1, 0, s>>>( A ); LAUNCHED();
		uint32_t num = n > HQ_SMALL ? 1 : 0, level = 0, max_count = n, max_cluster = HQ_MAX_CLUSTER;
		CUDA_TRY( cudaFuncSetAttribute( k_hq_level, cudaFuncAttributeNonPortableClusterSizeAllowed, 1 ) ); // clusters of more than 8 CTAs
		while (num)
		{
			CUDA_TRY( cudaMemsetAsync( &A.ctr->next_big, 0, 8, s ) ); // next_big + next_max
			// cluster size: enough CTAs for the largest node of the level, at most 8 CTAs per SM in flight (constants measured on B200,
			// profiles/README.md)
			uint32_t nct = 1;
			while (nct < max_cluster && (size_t)nct * HQ_CTA_FRAGS < max_count && (size_t)num * nct * 2 <= (size_t)b->ctx->sm_count * HQ_CTA_CAP) nct <<= 1;
			cudaLaunchConfig_t cfg = {};
			cudaLaunchAttribute attr[1];
			cfg.gridDim = dim3( num * nct ), cfg.blockDim = dim3( HQ_BIG_THREADS ), cfg.dynamicSmemBytes = 0, cfg.stream = s;
			attr[0].id = cudaLaunchAttributeClusterDimension, attr[0].val.clusterDim.x = nct, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
			cfg.attrs = attr, cfg.numAttrs = 1;
			{
				// a cluster shape the device cannot co-schedule (MIG slices, fewer SMs per GPC) fails at launch: nothing has run, so
				// fall back to the next smaller shape
				const cudaError_t le = cudaLaunchKernelEx( &cfg, k_hq_level, A, (const HQTask*)A.lvl[level & 1], A.lvl[(level + 1) & 1], nct );
				if (le != cudaSuccess && nct > 1) { cudaGetLastError(); max_cluster = nct >> 1; continue; }
				CUDA_TRY( le ); LAUNCHED();
			}
			CUDA_TRY( cudaMemcpyAsync( h_ctr, A.ctr, sizeof( HQCounters ), cudaMemcpyDeviceToHost, s ) );
			CUDA_TRY( cudaStreamSynchronize( s ) );
			if (A.profile > 1)
			{
				static unsigned long long prev[12];
				if (level == 0) memset( prev, 0, sizeof( prev ) );
				fprintf( stderr, "hq-level %2u nodes %5u nct %2u max %7u:", level, num, nct, max_count );
				for (int k = 0; k < 12; k++) { fprintf( stderr, " %7.1f", (h_ctr->prof[k] - prev[k]) * 1e-3 / num ); prev[k] = h_ctr->prof[k]; }
				fprintf( stderr, "  kcyc/node\n" );
			}
			num = h_ctr->next_big, max_count = h_ctr->next_max;
			if (h_ctr->overflow) { tbvh_set_error( "BuildHQ: pool overflow in the level phase" ); return TBVH_E_LIMIT; }
			if (++level > 4096) { tbvh_set_error( "BuildHQ: runaway level count" ); return TBVH_E_LIMIT; }
		}
		CUDA_TRY( cudaMemcpyAsync( h_ctr, A.ctr, sizeof( HQCounters ), cudaMemcpyDeviceToHost, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		const uint32_t roots = h_ctr->small_roots;
		if (roots) { k_hq_subtrees<<<(roots + HQ_SMALL_WARPS - 1) / HQ_SMALL_WARPS, HQ_SMALL_WARPS * 32, 0, s>>>( A, roots ); LAUNCHED(); }
		CUDA_TRY( cudaMemcpyAsync( h_ctr, A.ctr, sizeof( HQCounters ), cudaMemcpyDeviceToHost, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		if (h_ctr->overflow) { tbvh_set_error( "BuildHQ: pool overflow in the subtree phase" ); return TBVH_E_LIMIT; }
		const uint32_t tmp_count = h_ctr->node_ptr;
		if (A.profile)
		{
			static const char* nm[12] = { "obj-bin", "obj-sweep", "spat-bin", "spat-sweep", "part-obj", "part-p1", "chain", "split", "p4+bounds", "leaf", "copyback", "emit" };
			for (int k = 0; k < 12; k++) fprintf( stderr, "hq-profile %-10s level %10.3f Mcyc   subtree %10.3f Mcyc\n", nm[k], h_ctr->prof[k] * 1e-6, h_ctr->prof[16 + k] * 1e-6 );
			fprintf( stderr, "hq-profile failed_splits %u small_roots %u\n", h_ctr->failed_splits, h_ctr->small_roots );
		}
		// Compact(): DFS-preorder numbering, leaf index ranges packed in DFS order; the tail of the index array is zeroed
		CUDA_TRY( cudaMemsetAsync( b->d_prim_idx, 0, (size_t)A.idx_cap * 4, s ) );
		if (tmp_count > 2)
		{
			k_hq_up<<<(tmp_count + 255) / 256, 256, 0, s>>>( A, tmp_count ); LAUNCHED();
			k_hq_down<<<(tmp_count + 255) / 256, 256, 0, s>>>( A, tmp_count, b->d_nodes, b->d_prim_idx ); LAUNCHED();
		}
		else
		{
			CUDA_TRY( cudaMemcpyAsync( b->d_nodes, A.tmp_nodes, 64, cudaMemcpyDeviceToDevice, s ) );
			CUDA_TRY( cudaMemcpyAsync( b->d_prim_idx, A.prim_idx, (size_t)A.idx_cap * 4, cudaMemcpyDeviceToDevice, s ) );
		}
		CUDA_TRY( cudaEventRecord( e1, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		float ms = 0;
		CUDA_TRY( cudaEventElapsedTime( &ms, e0, e1 ) );
		b->info.build_ms = ms;
		b->info.used_nodes = tmp_count, b->info.idx_count = A.idx_cap, b->info.max_depth = h_ctr->max_depth;
		uint32_t rootw[8];
		CUDA_TRY( cudaMemcpy( rootw, b->d_nodes, 32, cudaMemcpyDeviceToHost ) );
		memcpy( b->info.aabb_min, rootw, 12 ), memcpy( b->info.aabb_max, rootw + 4, 12 );
		b->root_ref = rootw[3], b->root_count = rootw[7];
		b->d_trav = b->d_nodes;
		return make_leaf_tris( b, s );
	};
	const int rc = body();
	cudaStreamSynchronize( s );
	for (void* p : scratch) cudaFree( p );
	if (h_ctr) cudaFreeHost( h_ctr );
	if (e0) cudaEventDestroy( e0 );
	if (e1) cudaEventDestroy( e1 );
	return rc;
}
