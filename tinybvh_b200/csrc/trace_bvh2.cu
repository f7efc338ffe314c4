// tinybvh_b200/csrc/trace_bvh2.cu - BVH2 closest-hit / any-hit traversal for sm_100a.
//
// Replaces BVH::Intersect<posX,posY,posZ> (tiny_bvh.h:3247-3304), BVH::IsOccluded<...> (:3407-3453) and the OpenCL
// kernels traverse_ailalaine / isoccluded_ailalaine (traverse_bvh2.cl:80,147) for whole ray batches.
//
// Semantics are the oracle's, bit for bit (SURVEY.md Appendix A): stored rD, slab term fma(bound, rD, -(O*rD)),
// tmin = max(tx1,ty1,tz1,0), tmax = min(tx2,ty2,tz2,hit.t), hit iff tmax >= tmin, nearer child first with the LEFT
// child on ties, leaf triangles in primIdx order, Moeller-Trumbore accepted on t in [0, hit.t] (later equal-t hits win).
//
// Device layout (DESIGN.md "BVH2 in HBM"): the two children of an interior node are one 64-byte, 64-aligned record
// (the reference's sibling pair nodes[leftFirst], nodes[leftFirst+1]) fetched as 4 x LDG.128; a child is
// {min.xyz, ref, max.xyz, count}: count == 0 -> interior, ref = index of its own pair; count > 0 -> leaf, ref = first
// record in the leaf-ordered triangle array (3 x float4 per triangle: v0|primIdx, e1, e2), so a leaf costs no node
// fetch and no primIdx indirection.
#include "common.cuh"
#include <stdlib.h>

// SLAB_TEST_TWO_NODES (tiny_bvh.h:3202-3220) for the child pair (a, b): near plane = min when D >= 0 else max.
// The octant flags are compile-time in the specialised instances (no selects) and run-time in the generic one.
#define SLAB_PAIR( PX, PY, PZ ) \
	const float tx1a = __fmaf_rn( (PX) ? a0.x : a1.x, rdx, nrox ), tx2a = __fmaf_rn( (PX) ? a1.x : a0.x, rdx, nrox ); \
	const float ty1a = __fmaf_rn( (PY) ? a0.y : a1.y, rdy, nroy ), ty2a = __fmaf_rn( (PY) ? a1.y : a0.y, rdy, nroy ); \
	const float tz1a = __fmaf_rn( (PZ) ? a0.z : a1.z, rdz, nroz ), tz2a = __fmaf_rn( (PZ) ? a1.z : a0.z, rdz, nroz ); \
	const float tx1b = __fmaf_rn( (PX) ? b0.x : b1.x, rdx, nrox ), tx2b = __fmaf_rn( (PX) ? b1.x : b0.x, rdx, nrox ); \
	const float ty1b = __fmaf_rn( (PY) ? b0.y : b1.y, rdy, nroy ), ty2b = __fmaf_rn( (PY) ? b1.y : b0.y, rdy, nroy ); \
	const float tz1b = __fmaf_rn( (PZ) ? b0.z : b1.z, rdz, nroz ), tz2b = __fmaf_rn( (PZ) ? b1.z : b0.z, rdz, nroz ); \
	tmina = fmaxf( fmaxf( tx1a, ty1a ), fmaxf( tz1a, 0.0f ) ), tminb = fmaxf( fmaxf( tx1b, ty1b ), fmaxf( tz1b, 0.0f ) ); \
	tmaxa = fminf( fminf( tx2a, ty2a ), fminf( tz2a, tmax ) ), tmaxb = fminf( fminf( tx2b, ty2b ), fminf( tz2b, tmax ) );

// 10 resident CTAs per SM asked of ptxas: 40 warps / SM without spills (12 and 16 were measured slower).
// OCTSW = 1: when every ray of the warp lies in the same direction octant (the normal case for camera and shadow rays) the
// slab tests run through an octant-specialised instance picked by a warp-uniform switch, which removes the 12 selects
// per step; mixed warps use the generic per-lane selects.  Same arithmetic, same order, same results either way.
// STACKN = traversal stack entries: TBVH_STACK (64) for trees of depth < 64, TBVH_STACK_DEEP (256, the reference's own stack, :3249) above.
template <bool ANYHIT, bool STATS, int OCTSW, int STACKN>
__global__ void __launch_bounds__( 128, 10 ) k_trace_bvh2( const float4* __restrict__ nodes, const float4* __restrict__ tris,
	const char* rays, const uint32_t stride, char* hits, const uint32_t hit_stride, // may alias (in-place hits): plain loads
	uint32_t* __restrict__ bits, const uint64_t n, const uint32_t root_ref, const uint32_t root_count,
	unsigned long long* __restrict__ stats )
{
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	bool occluded = false;
	const bool valid = i < n;
	float4 ro4 = make_float4( 0, 0, 0, 0 ), rd4 = ro4, rr4 = ro4, rh4 = ro4;
	if (valid)
	{
		const float4* rp = (const float4*)(rays + i * stride);
		ro4 = rp[0], rd4 = rp[1], rr4 = rp[2], rh4 = rp[3];
	}
	const bool posX = rd4.x >= 0, posY = rd4.y >= 0, posZ = rd4.z >= 0;
	const uint32_t oct = (posX ? 4u : 0u) | (posY ? 2u : 0u) | (posZ ? 1u : 0u);
	bool uni = false;
	if (OCTSW)
	{
		const uint32_t vm = __ballot_sync( 0xffffffffu, valid );
		const uint32_t oct0 = __shfl_sync( 0xffffffffu, oct, vm ? __ffs( vm ) - 1 : 0 );
		uni = __all_sync( 0xffffffffu, !valid || oct == oct0 );
	}
	if (valid)
	{
		const float ox = ro4.x, oy = ro4.y, oz = ro4.z, dx = rd4.x, dy = rd4.y, dz = rd4.z;
		const float rdx = rr4.x, rdy = rr4.y, rdz = rr4.z;
		// -(O*rD), rounded product as the oracle's `rox` (:3252-3254)
		const float nrox = -__fmul_rn( ox, rdx ), nroy = -__fmul_rn( oy, rdy ), nroz = -__fmul_rn( oz, rdz );
		float tmax = rh4.x, hu = rh4.y, hv = rh4.z;
		uint32_t hprim = __float_as_uint( rh4.w );
		uint2 stack[STACKN];
		int sp = 0;
		uint32_t ref = root_ref, cnt = root_count;
		unsigned long long nsteps = 0, ntris = 0;
		while (true)
		{
			if (STATS) nsteps++;
			if (cnt == 0)
			{
				// interior: fetch the 64-byte child pair
				const float4* p = nodes + (size_t)ref * 2;
				const float4 a0 = __ldg( p ), a1 = __ldg( p + 1 ), b0 = __ldg( p + 2 ), b1 = __ldg( p + 3 );
				float tmina, tminb, tmaxa, tmaxb;
				if (OCTSW && uni)
				{
					switch (oct)
					{
					case 0: { SLAB_PAIR( false, false, false ) } break;
					case 1: { SLAB_PAIR( false, false, true ) } break;
					case 2: { SLAB_PAIR( false, true, false ) } break;
					case 3: { SLAB_PAIR( false, true, true ) } break;
					case 4: { SLAB_PAIR( true, false, false ) } break;
					case 5: { SLAB_PAIR( true, false, true ) } break;
					case 6: { SLAB_PAIR( true, true, false ) } break;
					default: { SLAB_PAIR( true, true, true ) } break;
					}
				}
				else { SLAB_PAIR( posX, posY, posZ ) }
				const bool hita = tmaxa >= tmina, hitb = tmaxb >= tminb;
				const uint32_t refa = __float_as_uint( a0.w ), cnta = __float_as_uint( a1.w );
				const uint32_t refb = __float_as_uint( b0.w ), cntb = __float_as_uint( b1.w );
				if (hita && hitb)
				{
					// swap only on dist1 > dist2: ties visit the left child first (:3292)
					const bool swp = tmina > tminb;
					ref = swp ? refb : refa, cnt = swp ? cntb : cnta;
					stack[sp++] = swp ? make_uint2( refa, cnta ) : make_uint2( refb, cntb );
					continue;
				}
				if (hita) { ref = refa, cnt = cnta; continue; }
				if (hitb) { ref = refb, cnt = cntb; continue; }
			}
			else
			{
				// leaf: cnt triangles starting at record ref, in primIdx order (:3281-3285)
				const float4* tp = tris + (size_t)ref * 3;
				for (uint32_t k = 0; k < cnt; k++, tp += 3)
				{
					const float4 v0 = __ldg( tp ), e1 = __ldg( tp + 1 ), e2 = __ldg( tp + 2 );
					float t, u, v;
					if (STATS) ntris++;
					if (mt_test( ox, oy, oz, dx, dy, dz, v0, e1, e2, tmax, t, u, v ))
					{
						if (ANYHIT) { occluded = true; break; }
						tmax = t, hu = u, hv = v, hprim = __float_as_uint( v0.w );
					}
				}
				if (ANYHIT && occluded) break;
			}
			if (sp == 0) break;
			const uint2 e = stack[--sp];
			ref = e.x, cnt = e.y;
		}
		if (!ANYHIT)
		{
			float4* hp = (float4*)(hits + i * hit_stride);
			*hp = make_float4( tmax, hu, hv, __uint_as_float( hprim ) );
		}
		if (STATS) { atomicAdd( &stats[0], nsteps ); atomicAdd( &stats[1], ntris ); }
	}
	if (ANYHIT)
	{
		// blockDim is a multiple of 32 and i is the global thread index: lane l of a warp holds ray 32*w + l
		const uint32_t m = __ballot_sync( 0xffffffffu, occluded );
		if ((threadIdx.x & 31) == 0 && (i & ~31ull) < n) bits[i >> 5] = m;
	}
}

int bvh2_trace_launch( tbvh_bvh b, const void* d_rays, uint32_t stride, void* d_hits, uint32_t hit_stride, uint32_t* d_bits,
	uint64_t n, bool anyhit, cudaStream_t s, unsigned long long* d_stats )
{
	if (!b->d_trav || !b->d_leaf_tris) { tbvh_set_error( "BVH2 layout not resident" ); return TBVH_E_STATE; }
	if (n == 0) return TBVH_OK;
	if (b->info.max_depth + 1 > TBVH_STACK_DEEP) { tbvh_set_error( "BVH depth %u exceeds the %d-entry traversal stack (the reference's own, tiny_bvh.h:3249)", b->info.max_depth, TBVH_STACK_DEEP ); return TBVH_E_LIMIT; }
	const bool deep = b->info.max_depth + 1 > TBVH_STACK;
	const uint32_t root_ref = b->root_ref, root_count = b->root_count;
	const uint32_t block = 128;
	const uint64_t grid = (n + block - 1) / block;
	if (grid > 0x7fffffffull) { tbvh_set_error( "ray batch too large for one launch" ); return TBVH_E_ARG; }
	// statistics launches run the per-lane slab step (OCTSW = 0), every other launch the octant switch
	#define LAUNCH( A, S, O, D ) k_trace_bvh2<A, S, O, D><<<(uint32_t)grid, block, 0, s>>>( b->d_trav, b->d_leaf_tris, (const char*)d_rays, stride, \
		(char*)d_hits, hit_stride, d_bits, n, root_ref, root_count, d_stats )
	if (deep)
	{
		// depth 64..255: the same kernel with the reference's 256-entry stack (2 KiB of local memory per ray)
		if (d_stats) { if (anyhit) LAUNCH( true, true, 0, TBVH_STACK_DEEP ); else LAUNCH( false, true, 0, TBVH_STACK_DEEP ); }
		else { if (anyhit) LAUNCH( true, false, 1, TBVH_STACK_DEEP ); else LAUNCH( false, false, 1, TBVH_STACK_DEEP ); }
	}
	else if (d_stats) { if (anyhit) LAUNCH( true, true, 0, TBVH_STACK ); else LAUNCH( false, true, 0, TBVH_STACK ); }
	else { if (anyhit) LAUNCH( true, false, 1, TBVH_STACK ); else LAUNCH( false, false, 1, TBVH_STACK ); }
	#undef LAUNCH
	LAUNCHED();
	return TBVH_OK;
}
