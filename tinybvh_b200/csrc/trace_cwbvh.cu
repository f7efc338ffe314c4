// tinybvh_b200/csrc/trace_cwbvh.cu - closest-hit / any-hit traversal of BVH8_CWBVH data on sm_100a.
//
// Results are those of the reference's own walk of the same data, BVH8_CWBVH::Intersect (tiny_bvh.h:7046-7154), bit for bit:
// children of a wide node are entered in the order the format defines (inner child in slot s owns bit 24 + (s ^ o) of the
// node's hit word, o = 7 - ray octant; highest bit first), a leaf child owns `count` consecutive bits from its triangle offset,
// a child is hit iff  max( tnear_x, tnear_y, tnear_z, 0 ) <= min( tfar_x, tfar_y, tfar_z, t )  with
// t_plane = fma( q, 2^e * rD, ( p - O ) * rD ),  triangles run through the oracle's Moeller-Trumbore (common.cuh mt_test).
//
// What is different from the reference kernels (traverse_cwbvh.cl) is everything the format does not dictate:
//
//  * The kernels do not read bvh8Data.  `cw_make_trav` expands every 80-byte node once into a 160-byte TRAVERSAL NODE made for
//    this GPU (ncu on the byte format: 79 % issue-slot use, ALU pipe 72 % busy, 370 instructions per node visit, of which 96
//    turn bytes into floats and ~90 test slots that hold no child - the reference's 8-wide collapse fills 4.4 of 8 slots on
//    Bistro, 36 % of the nodes have two children):
//        header   32 B   p.xyz | 2^ex 2^ey as float top halves | first inner child | first triangle (float4 units) | 2^ez, imask, pairs | children
//        pair j   32 B   the (2j)-th and (2j+1)-th NON-EMPTY child:  lo.x lo.y lo.z hi.x hi.y hi.z as half2 (child a, child b)
//                        - 0..255 is exact in fp16 - and one 32-bit hit word per child: a leaf child's triangle bits
//                        `unary(count) << offset`, an inner child's slot bit `1 << (24 + slot)`
//    Empty slots are gone: a node holds ceil(children/2) pair records (the rest of the four are zero and contribute no bit), and a
//    visited node is nearly always full (3.83 of 4 on Bistro camera rays), so the kernel runs all four pair steps without branching -
//    four pair steps instead of eight slot steps, and the eight loads leave together.
//  * A pair step is packed fp32 arithmetic (Blackwell FFMA2, `fma.rn.f32x2`): one instruction evaluates the same plane of both
//    children, 6 per pair instead of 12 FFMA, exactly rounded per component like the scalar fma.
//  * The quantised planes reach the registers as halves and are widened by one conversion each (no byte extraction, no
//    integer-to-float on the quarter-rate unit, no magic-number subtraction).
//  * Near / far planes are picked by the sign of rD once per pair on the packed words, inner-child bits are accumulated in slot order
//    and moved to octant order by one 3-stage bit butterfly per node - and when every ray of a warp points into the same direction
//    octant (camera and shadow rays), a warp-uniform switch runs the node step through the instance compiled for that octant, where
//    both are compile-time (node_hits<OCT>).
//  * The per-axis scales 2^e are stored as the top halves of their float patterns: one shift or mask each instead of a byte decode.
//
// Executed-instruction mix, ncu extracts and the history of the variants: profiles/README.md ("The CWBVH kernel ...").
//
// Triangles are the reference's 48-byte records (e2, e1, v0 | primIdx) read straight from bvh8Tris.
#include "cw_walk.cuh"
#include <vector>

// ---- bvh8Data -> traversal nodes ------------------------------------------------------------------------------------
// One thread per node.  Slot i of the source node: meta byte i (n1.z / n1.w), quantised bounds byte i of the six 8-byte rows at
// bytes 32..79 (lo.x, lo.y, lo.z, hi.x, hi.y, hi.z) - layout in SURVEY.md 8(a), written by BVH8_CWBVH::ConvertFrom (tiny_bvh.h:5948-6015).
__global__ void k_cw_expand( const uint4* __restrict__ src, uint4* __restrict__ dst, uint32_t* __restrict__ parent, const uint32_t count )
{
	const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
	if (x >= count) return;
	const uint4 n0 = src[(size_t)x * 5], n1 = src[(size_t)x * 5 + 1], n2 = src[(size_t)x * 5 + 2], n3 = src[(size_t)x * 5 + 3], n4 = src[(size_t)x * 5 + 4];
	const uint32_t row[6][2] = { { n2.x, n2.y }, { n2.z, n2.w }, { n3.x, n3.y }, { n3.z, n3.w }, { n4.x, n4.y }, { n4.z, n4.w } };
	const uint32_t meta[2] = { n1.z, n1.w };
	uint32_t word[4][8]; // pair records under construction
	#pragma unroll
	for (int j = 0; j < 4; j++) for (int k = 0; k < 8; k++) word[j][k] = 0;
	uint32_t kept = 0, inner = 0;
	#pragma unroll
	for (int i = 0; i < 8; i++)
	{
		const uint32_t m = (meta[i >> 2] >> (8 * (i & 3))) & 255u;
		if (m == 0) continue; // empty slot: contributes no bit whatever its box test says
		const bool is_inner = (m & 0x18u) == 0x18u; // 0b001sssss with sssss = 24 + slot (tiny_bvh.h:5988); a triangle offset is < 24
		const uint32_t bits = is_inner ? 1u << (24u + (m & 7u)) : (m >> 5) << (m & 31u);
		if (is_inner) inner++;
		const uint32_t j = kept >> 1, side = kept & 1;
		#pragma unroll
		for (int r = 0; r < 6; r++)
		{
			const uint32_t q = (row[r][i >> 2] >> (8 * (i & 3))) & 255u;
			const uint32_t h = CW_PLANES_BF16 ? __float_as_uint( (float)q ) >> 16 : (uint32_t)__half_as_ushort( __uint2half_rn( q ) );
			#pragma unroll
			for (int jj = 0; jj < 4; jj++) if (jj == (int)j) word[jj][r] |= side ? h << 16 : h;
		}
		#pragma unroll
		for (int jj = 0; jj < 4; jj++) if (jj == (int)j) word[jj][6 + side] = bits;
		kept++;
	}
	uint4* o = dst + (size_t)x * CW_NODE_F4;
	// 2^e per axis as the top half of its float bit pattern, ( e + 127 ) << 7 for the signed exponent byte e - including the
	// reference's own wrap for e = -128, ( -1 ) << 23 = 0xff800000 (tiny_bvh.h:7072-7074)
	const uint32_t sx = (uint32_t)(((int)(int8_t)(n0.w & 255u) + 127) * 128) & 0xffffu, sy = (uint32_t)(((int)(int8_t)((n0.w >> 8) & 255u) + 127) * 128) & 0xffffu;
	const uint32_t sz = (uint32_t)(((int)(int8_t)((n0.w >> 16) & 255u) + 127) * 128) & 0xffffu;
	o[0] = make_uint4( n0.x, n0.y, n0.z, sx | (sy << 16) );
	o[1] = make_uint4( n1.x, n1.y, sz | ((n0.w >> 24) << 16) | (((kept + 1) >> 1) << 24), kept );
	#pragma unroll
	for (int j = 0; j < 4; j++)
	{
		o[2 + 2 * j] = make_uint4( word[j][0], word[j][1], word[j][2], word[j][3] );
		o[3 + 2 * j] = make_uint4( word[j][4], word[j][5], word[j][6], word[j][7] );
	}
	// inner children sit at n1.x + 0 .. inner-1 (node units): note their parent for the depth pass
	if (parent) for (uint32_t c = 0; c < inner; c++) if (n1.x + c < count) parent[n1.x + c] = x;
}

__global__ void k_cw_depth( const uint32_t* __restrict__ parent, const uint32_t count, uint32_t* __restrict__ max_depth )
{
	const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
	if (x >= count) return;
	uint32_t d = 0, n = x;
	while (n != 0 && n < count && d < 4096) n = parent[n], d++; // n >= count: a record no node points at (0xffffffff)
	if (n != 0) return;
	atomicMax( max_depth, d );
}

int cw_make_trav( tbvh_bvh b, cudaStream_t s, int known_depth )
{
	if (b->d_cw_trav) cudaFree( b->d_cw_trav ), b->d_cw_trav = 0;
	const uint32_t count = b->info.used_blocks / 5;
	if (count == 0) { tbvh_set_error( "cw_make_trav: no CWBVH nodes" ); return TBVH_E_STATE; }
	CUDA_TRY( cudaMalloc( &b->d_cw_trav, (size_t)count * CW_NODE_F4 * 16 ) );
	if (known_depth >= 0)
	{
		k_cw_expand<<<(count + 127) / 128, 128, 0, s>>>( (const uint4*)b->d_cw_nodes, (uint4*)b->d_cw_trav, 0, count ); LAUNCHED();
		b->cw_depth = (uint32_t)known_depth;
		return TBVH_OK;
	}
	// uploaded data: the depth of the wide tree is not known - every node notes its parent, then walks up to the root
	uint32_t* d_parent = 0;
	CUDA_TRY( cudaMalloc( &d_parent, ((size_t)count + 1) * 4 ) );
	uint32_t depth = 0;
	auto body = [&]() -> int
	{
		CUDA_TRY( cudaMemsetAsync( d_parent, 0xff, (size_t)count * 4, s ) );
		CUDA_TRY( cudaMemsetAsync( d_parent + count, 0, 4, s ) );
		k_cw_expand<<<(count + 127) / 128, 128, 0, s>>>( (const uint4*)b->d_cw_nodes, (uint4*)b->d_cw_trav, d_parent, count ); LAUNCHED();
		k_cw_depth<<<(count + 127) / 128, 128, 0, s>>>( d_parent, count, d_parent + count ); LAUNCHED();
		CUDA_TRY( cudaMemcpyAsync( &depth, d_parent + count, 4, cudaMemcpyDeviceToHost, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		return TBVH_OK;
	};
	const int rc = body();
	cudaFree( d_parent );
	b->cw_depth = depth;
	return rc;
}

// ---- traversal ------------------------------------------------------------------------------------------------------

// OCTSW = 1: warps whose rays all point into one direction octant (camera and shadow rays: nearly all of them) run the node step
// through the instance compiled for that octant, picked by a warp-uniform switch; mixed warps use the per-lane form.
template <bool ANYHIT, bool STATS, int OCTSW>
__global__ void __launch_bounds__( 128 ) k_trace_wide( const float4* __restrict__ nodes, const float4* __restrict__ tris,
	const char* rays, const uint32_t stride, char* hits, const uint32_t hit_stride, uint32_t* __restrict__ bits, const uint64_t n,
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
	const float ox = ro4.x, oy = ro4.y, oz = ro4.z, dx = rd4.x, dy = rd4.y, dz = rd4.z;
	const float rdx = rr4.x, rdy = rr4.y, rdz = rr4.z;
	const uint32_t o = 7u - ((dx < 0 ? 4u : 0u) | (dy < 0 ? 2u : 0u) | (dz < 0 ? 1u : 0u)); // octinv of tiny_bvh.h:7053 (signs of D)
	const bool negx = rdx < 0, negy = rdy < 0, negz = rdz < 0;                                // plane swizzle uses rD (:7082)
	const uint32_t oct = (negx ? 4u : 0u) | (negy ? 2u : 0u) | (negz ? 1u : 0u);
	bool uni = false;
	if (OCTSW)
	{
		// the compiled-in octant serves both the plane choice (signs of rD) and the visiting order (signs of D): they must agree
		const uint32_t vm = __ballot_sync( 0xffffffffu, valid );
		const uint32_t oct0 = __shfl_sync( 0xffffffffu, oct, vm ? __ffs( vm ) - 1 : 0 );
		uni = __all_sync( 0xffffffffu, !valid || (oct == oct0 && o == 7u - oct) );
	}
	if (valid)
	{
		float t = rh4.x, hu = rh4.y, hv = rh4.z;
		uint32_t hprim = __float_as_uint( rh4.w );
		uint2 pending[CW_STACK];
		int depth = 0;
		uint32_t base = 0, word = 0x80000000u; // the root as a one-child group: bit 31, no siblings
		unsigned long long nsteps = 0, ntris = 0, npairs = 0;
		while (true)
		{
			// ---- enter the pending inner child with the highest bit
			const uint32_t bit = 31u - __clz( word );
			const uint32_t rest = word & ~(1u << bit);
			if (rest > 0x00ffffffu) pending[depth++] = make_uint2( base, rest );
			const uint32_t slot = (bit - 24u) ^ o;
			const uint32_t nidx = base + __popc( word & ~(0xffffffffu << slot) );
			const float4* np = nodes + (size_t)nidx * CW_NODE_F4;
			const float4 h0 = __ldg( np ), h1 = __ldg( np + 1 );
			if (STATS) nsteps++;
			// scale = 2^e as a float bit pattern, ( e + 127 ) << 23 (:7072-7074), stored by cw_make_trav as top halves
			const uint32_t sxy = __float_as_uint( h0.w ), szm = __float_as_uint( h1.z );
			const float scx = __uint_as_float( sxy << 16 ), scy = __uint_as_float( sxy & 0xffff0000u ), scz = __uint_as_float( szm << 16 );
			const float ax1 = __fmul_rn( scx, rdx ), ay1 = __fmul_rn( scy, rdy ), az1 = __fmul_rn( scz, rdz );
			const float bx1 = __fmul_rn( -__fsub_rn( ox, h0.x ), rdx ), by1 = __fmul_rn( -__fsub_rn( oy, h0.y ), rdy ), bz1 = __fmul_rn( -__fsub_rn( oz, h0.z ), rdz );
			const uint32_t pairs = szm >> 24;
			if (STATS) npairs += pairs;
			uint32_t got;
			#define NODE_HITS( O ) got = node_hits<O>( np, pairs, negx, negy, negz, o, ax1, ay1, az1, bx1, by1, bz1, t )
			if (OCTSW && uni)
			{
				switch (oct)
				{
				case 0: NODE_HITS( 0 ); break;
				case 1: NODE_HITS( 1 ); break;
				case 2: NODE_HITS( 2 ); break;
				case 3: NODE_HITS( 3 ); break;
				case 4: NODE_HITS( 4 ); break;
				case 5: NODE_HITS( 5 ); break;
				case 6: NODE_HITS( 6 ); break;
				default: NODE_HITS( 7 ); break;
				}
			}
			else NODE_HITS( -1 );
			#undef NODE_HITS
			base = __float_as_uint( h1.x );
			word = (got & 0xff000000u) | ((szm >> 16) & 255u);
			// ---- triangles of the leaf children that were hit, highest bit first (:7132-7142)
			uint32_t tmask = got & 0x00ffffffu;
			const float4* tbase = tris + __float_as_uint( h1.y );
			while (tmask)
			{
				const uint32_t k = 31u - __clz( tmask );
				tmask &= ~(1u << k);
				const float4* tp = tbase + k * 3;
				const float4 e2 = __ldg( tp ), e1 = __ldg( tp + 1 ), v0 = __ldg( tp + 2 );
				if (STATS) ntris++;
				float tt, u, v;
				if (mt_test( ox, oy, oz, dx, dy, dz, v0, e1, e2, t, tt, u, v ))
				{
					if (ANYHIT) { occluded = true; break; }
					t = tt, hu = u, hv = v, hprim = __float_as_uint( v0.w );
				}
			}
			if (ANYHIT && occluded) break;
			if (word > 0x00ffffffu) continue;
			if (depth == 0) break;
			const uint2 e = pending[--depth];
			base = e.x, word = e.y;
		}
		if (!ANYHIT)
		{
			float4* hp = (float4*)(hits + i * hit_stride);
			*hp = make_float4( t, hu, hv, __uint_as_float( hprim ) );
		}
		if (STATS) { atomicAdd( &stats[0], nsteps ); atomicAdd( &stats[1], ntris ); atomicAdd( &stats[2], npairs ); }
	}
	if (ANYHIT)
	{
		const uint32_t m = __ballot_sync( 0xffffffffu, occluded );
		if ((threadIdx.x & 31) == 0 && (i & ~31ull) < n) bits[i >> 5] = m;
	}
}

int cwbvh_trace_launch( tbvh_bvh b, const void* d_rays, uint32_t stride, void* d_hits, uint32_t hit_stride, uint32_t* d_bits,
	uint64_t n, bool anyhit, cudaStream_t s, unsigned long long* d_stats )
{
	if (!b->d_cw_trav || !b->d_cw_tris) { tbvh_set_error( "CWBVH layout not resident" ); return TBVH_E_STATE; }
	if (n == 0) return TBVH_OK;
	if (b->cw_depth + 1 > CW_STACK) { tbvh_set_error( "wide-tree depth %u exceeds the %d pending node groups a ray can hold (the reference's own limit)", b->cw_depth, CW_STACK ); return TBVH_E_LIMIT; }
	const uint32_t block = 128;
	const uint64_t grid = (n + block - 1) / block;
	if (grid > 0x7fffffffull) { tbvh_set_error( "ray batch too large for one launch" ); return TBVH_E_ARG; }
	// statistics launches run the per-lane node step (OCTSW = 0), every other launch the octant switch
	#define LAUNCH( A, S, O ) k_trace_wide<A, S, O><<<(uint32_t)grid, block, 0, s>>>( b->d_cw_trav, b->d_cw_tris, (const char*)d_rays, stride, \
		(char*)d_hits, hit_stride, d_bits, n, d_stats )
	if (anyhit) { if (d_stats) LAUNCH( true, true, 0 ); else LAUNCH( true, false, 1 ); }
	else { if (d_stats) LAUNCH( false, true, 0 ); else LAUNCH( false, false, 1 ); }
	#undef LAUNCH
	LAUNCHED();
	return TBVH_OK;
}
