// tinybvh_b200/csrc/common.cuh - shared device/host definitions of the sm_100a engine.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <mutex>
#include <vector>
#include <atomic>
#include "../../include/tinybvh_b200.h"

#define BVH_FAR 1e30f
#define TBVH_STACK 64          // traversal stack entries per ray of the default BVH2 kernels; deeper trees run the TBVH_STACK_DEEP instances
#define TBVH_STACK_DEEP 256    // the reference's own closest-hit stack (tiny_bvh.h:3249; any-hit uses 64, :3409)

// ---- error plumbing -------------------------------------------------------------------------------------
void tbvh_set_error( const char* fmt, ... );
extern unsigned long long g_tbvh_launches;
#define CUDA_TRY( x ) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { tbvh_set_error( "%s:%d %s -> %s", __FILE__, __LINE__, #x, cudaGetErrorString( e_ ) ); return TBVH_E_CUDA; } } while (0)
#define LAUNCHED() do { g_tbvh_launches++; cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) { tbvh_set_error( "%s:%d launch -> %s", __FILE__, __LINE__, cudaGetErrorString( e_ ) ); return TBVH_E_CUDA; } } while (0)

// ---- handles ----------------------------------------------------------------------------------------------
// one stage buffer set of the host-buffer pipeline (api.cu "host path")
struct HostSlot
{
	void* d_rays = 0;                // chunk of 64-byte device records
	void* d_hits = 0;                // packed 16-byte hits of the chunk
	void* d_bits = 0;                // occlusion words of the chunk
	cudaEvent_t in_done = 0, run_done = 0, out_done = 0;
};
#define TBVH_SLOTS 4
#define TBVH_CHUNK_RAYS (1u << 19)   // rays per pipeline chunk (32 MiB of device records; 2^18 and 2^20 measured no better, profiles/README.md)

struct tbvh_ctx_t
{
	int device = 0;
	int sm_count = 148;
	cudaStream_t stream = 0;         // engine stream (builds, uploads, conversions)
	// host-buffer pipeline: inbound copies, traversal and outbound copies each own a stream, so chunk k+1 flows in while chunk k
	// is traced and the hits of chunk k-1 flow out; the slots are handed round-robin and recycled through events
	std::mutex host_mutex;           // host batch calls on one context are serialised (SURVEY 8(b): thread-safe per handle)
	cudaStream_t s_in = 0, s_run = 0, s_out = 0;
	HostSlot slot[TBVH_SLOTS];       // allocated by the first host batch call
	int inst_idx_bits = 32;          // the host program's INST_IDX_BITS (tiny_bvh.h:118): 32 = TLAS hits store hit.inst, 4..31 = top bits of hit.prim
	int small_t = 128;               // builder: subtrees of at most this many primitives go to the warp kernel (8..128; every value gives the same tree)
	int build_mode = 0;              // BVH::Build large phase: 0 = one persistent cooperative launch (k_large_phase), 1 = one launch per stage and level
};

uint32_t tbvh_next_generation(); // process-wide: a value no handle has carried before (a recycled handle address cannot revalidate a stale TLAS)
struct BlasLink { tbvh_bvh blas; uint32_t generation; }; // host side: what a TLAS was built over

struct tbvh_bvh_t
{
	tbvh_ctx ctx = 0;
	tbvh_info info = {};
	// geometry (engine-owned copy, float4 per vertex)
	float4* d_verts = 0;
	// LAYOUT_BVH: reference node array; children of an interior node are the 64-byte pair at nodes[leftFirst]
	float4* d_nodes = 0;       // 2 float4 per node
	uint32_t* d_prim_idx = 0;
	// traversal view of the BVH2: d_trav aliases d_nodes (LAYOUT_BVH) or is the pair array derived from a BVH_GPU upload
	float4* d_trav = 0;
	uint32_t root_ref = 0, root_count = 0; // the root as a child record: count==0 -> pair index, else leaf range
	// leaf-ordered triangle records for BVH2 traversal: 3 float4 per prim reference
	//   [0] = (v0.xyz, as_float(primIdx))  [1] = e1 = v1-v0  [2] = e2 = v2-v0
	float4* d_leaf_tris = 0;
	uint32_t leaf_tris_count = 0; // records d_leaf_tris was allocated for
	// LAYOUT_BVH_GPU mirror (only materialised on upload / convert / download)
	float4* d_nodes_gpu = 0;   // 4 float4 per node
	// LAYOUT_CWBVH
	float4* d_cw_nodes = 0;    // 5 float4 per node
	float4* d_cw_tris = 0;     // 3 float4 per triangle
	float4* d_cw_trav = 0;     // traversal nodes derived from d_cw_nodes (trace_cwbvh.cu cw_make_trav): 10 float4 per node
	uint32_t cw_depth = 0;     // depth of the wide tree (root = 0)
	uint32_t generation = 0;   // renewed (tbvh_next_generation) whenever the arrays a TLAS may point at are replaced (build, upload, refit, convert)
	// TLAS (BVH::Build( BLASInstance*, instCount, BVHBase**, blasCount ) :2221): nodes / primIdx over instance boxes + device tables
	float4* d_aabbs = 0;       // instance boxes the TLAS was built over (2 float4 per instance)
	void* d_inst = 0;          // TlasInst records (inverse transform, BLAS number, mask)
	void* d_blas = 0;          // BlasRef records (traversal arrays of every BLAS)
	uint32_t inst_count = 0, blas_count = 0;
	uint32_t tlas_blas_layouts = 0; // TLAS only: layouts EVERY BLAS held at build time (bit TBVH_LAYOUT_BVH / TBVH_LAYOUT_CWBVH)
	std::vector<BlasLink> links; // TLAS only: the BLAS handles it points into, with the generation they had at build time
	bool refittable = true;    // BVHBase::refittable (:811): false after BuildHQ ("can't refit an SBVH", :3027)
	// statistics
	int stats = 0;
	unsigned long long* d_stats = 0; // [0]=steps [1]=tris, accumulated over every launch of one API call
};

// ---- device math in the oracle's exact operation order (oracle/tbvh_oracle.c header lists the pairing) ----
// Every fused pair is spelled __fmaf_rn, every unfused product / sum an _rn intrinsic, so nvcc's own
// contraction (-fmad) cannot change the rounding.

// MOLLER_TRUMBORE_TEST tiny_bvh.h:1644-1656 with e1,e2 precomputed (identical bits: v1-v0 is exact-rounded once).
// Returns true when the triangle is accepted for [0, tmax]; writes t,u,v.
__device__ __forceinline__ bool mt_test( const float ox, const float oy, const float oz, const float dx, const float dy, const float dz,
	const float4 v0, const float4 e1, const float4 e2, const float tmax, float& t, float& u, float& v )
{
	const float hx = __fmaf_rn( dy, e2.z, -__fmul_rn( dz, e2.y ) );
	const float hy = __fmaf_rn( dz, e2.x, -__fmul_rn( dx, e2.z ) );
	const float hz = __fmaf_rn( dx, e2.y, -__fmul_rn( dy, e2.x ) );
	const float a = __fmaf_rn( e1.z, hz, __fmaf_rn( e1.x, hx, __fmul_rn( e1.y, hy ) ) );
	if (fabsf( a ) < 0.000001f) return false;
	const float f = __fdiv_rn( 1.0f, a );
	const float sx = __fsub_rn( ox, v0.x ), sy = __fsub_rn( oy, v0.y ), sz = __fsub_rn( oz, v0.z );
	u = __fmul_rn( f, __fmaf_rn( hz, sz, __fmaf_rn( hx, sx, __fmul_rn( hy, sy ) ) ) );
	const float qx = __fmaf_rn( -e1.y, sz, __fmul_rn( e1.z, sy ) );
	const float qy = __fmaf_rn( -e1.z, sx, __fmul_rn( e1.x, sz ) );
	const float qz = __fmaf_rn( -e1.x, sy, __fmul_rn( e1.y, sx ) );
	v = __fmul_rn( f, __fmaf_rn( dz, qz, __fmaf_rn( dy, qy, __fmul_rn( dx, qx ) ) ) );
	if (u < 0 || v < 0 || __fadd_rn( u, v ) > 1) return false;
	t = __fmul_rn( f, __fmaf_rn( e2.z, qz, __fmaf_rn( e2.x, qx, __fmul_rn( e2.y, qy ) ) ) );
	return !(t < 0 || t > tmax);
}

// order-preserving float <-> uint key for atomicMin/Max on floats
__device__ __forceinline__ uint32_t f2key( float f ) { uint32_t u = __float_as_uint( f ); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float key2f( uint32_t k ) { return __uint_as_float( (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k ); }

// ---- internal entry points (one per .cu) -------------------------------------------------------------------
// d_stats: NULL, or two counters the launch ADDS its node visits / triangle tests to (the caller zeroes them once per API call)
int bvh2_trace_launch( tbvh_bvh b, const void* d_rays, uint32_t stride, void* d_hits, uint32_t hit_stride, uint32_t* d_bits, uint64_t n, bool anyhit, cudaStream_t s, unsigned long long* d_stats );
int cwbvh_trace_launch( tbvh_bvh b, const void* d_rays, uint32_t stride, void* d_hits, uint32_t hit_stride, uint32_t* d_bits, uint64_t n, bool anyhit, cudaStream_t s, unsigned long long* d_stats );
int cw_make_trav( tbvh_bvh b, cudaStream_t s, int known_depth = -1 ); // known_depth < 0: measured on the device
int build_sah_launch( tbvh_bvh b, float c_trav, float c_int, int flavour );
int build_hq_launch( tbvh_bvh b, float c_trav, float c_int );
int refit_launch( tbvh_bvh b, cudaStream_t s );
int tlas_trace_launch( tbvh_bvh b, int layout, const void* d_rays, uint32_t stride, uint32_t* d_bits, uint64_t n, bool anyhit, cudaStream_t s );
struct TlasInst { float inv[16]; uint32_t blasIdx, mask, pad0, pad1; };                                  // 80 bytes
struct BlasRef { const float4* trav; const float4* tris; uint32_t root_ref, root_count, pad0, pad1; const float4* cw_nodes; const float4* cw_tris; }; // 48 bytes: BVH-layout arrays, CWBVH traversal nodes + bvh8Tris (0 when absent)
int make_leaf_tris( tbvh_bvh b, cudaStream_t s );
int bvh_gpu_to_bvh( tbvh_bvh b, uint32_t used_nodes_gpu, cudaStream_t s );
int bvh_to_bvh_gpu( tbvh_bvh b, cudaStream_t s );
int bvh_to_cwbvh( tbvh_bvh b, cudaStream_t s );
// exclusive scan of in[0..n) into out[0..n] (out[n] = total); tile_sum needs n/2048 + 2 words (build_sah.cu)
int exclusive_scan( const uint32_t* in, uint32_t* out, uint32_t* tile_sum, uint32_t n, cudaStream_t s );
