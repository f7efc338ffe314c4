/* include/tinybvh_b200.h - the drop-in boundary: a C-ABI over the B200 (sm_100a) engine.
 *
 * Plain pointers and sizes only; no torch / C++ types.  Each entry point names the reference interface it
 * replaces (file:line under the jbikker/tinybvh checkout, v1.6.7).  The C++ shim that keeps tinybvh's class
 * and method names on top of this ABI is include/tinybvh_b200.hpp; the reference-side binding a maintainer
 * would add is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every function returns TBVH_OK (0) or a negative TBVH_E_* code; tbvh_last_error() gives the message
 *    (the reference has no error codes: BVH_FATAL_ERROR prints and exit(1)s, tiny_bvh.h:1617-1620 - the
 *    shim maps non-zero to that behaviour).
 *  - there is NO CPU fallback: without a CUDA device every call that touches data fails with TBVH_E_CUDA.
 *  - `space` says where a caller pointer lives: TBVH_HOST or TBVH_DEVICE (device pointers are plain
 *    CUdeviceptr values of the context's device, e.g. torch tensor data_ptr()).
 *  - device-space INPUTS (vertices, indices, node arrays passed with TBVH_DEVICE) are read on the engine's own stream: the caller
 *    makes sure the work that produces them has completed (synchronise the producing stream) before the call.  The *_device
 *    traversal calls are the exception: they run on the stream the caller passes.
 *  - host batch calls (tbvh_intersect / _packed / tbvh_occluded) may be issued from several threads on one handle, as the
 *    reference's const Intersect / IsOccluded are (tiny_bvh_speedtest.cpp:392-401); they are serialised per context.  Builds,
 *    uploads, conversions and refits are exclusive, like the reference's Build.
 *  - ray records are the reference's `Ray` (tiny_bvh.h:688-709): O at byte 0, D at 16, rD at 32, hit
 *    (t,u,v,prim) at 48..63; `stride` is 128 for the host struct, 64 for the packed GPU record
 *    (traverse.cl:11-17).  hit.t on entry is the ray's maximum distance.
 */
#ifndef TINYBVH_B200_H
#define TINYBVH_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TBVH_OK 0
#define TBVH_E_CUDA -1      /* CUDA runtime / driver error, or no device */
#define TBVH_E_ARG -2       /* invalid argument */
#define TBVH_E_STATE -3     /* handle does not hold the requested layout */
#define TBVH_E_LIMIT -4     /* tree exceeds a device limit (e.g. depth > traversal stack) */
#define TBVH_E_UNSUPPORTED -5

#define TBVH_HOST 0
#define TBVH_DEVICE 1

/* layouts a handle can hold (values follow BVHBase::BVHType, tiny_bvh.h:773-793) */
#define TBVH_LAYOUT_BVH 1      /* Wald 32-byte nodes, BVH::BVHNode tiny_bvh.h:861-869 */
#define TBVH_LAYOUT_BVH_GPU 5  /* Aila-Laine 64-byte nodes, BVH_GPU::BVHNode tiny_bvh.h:1095-1105 */
#define TBVH_LAYOUT_CWBVH 10   /* 80-byte compressed wide nodes + 48-byte triangles, tiny_bvh.h:1356-1359 */

typedef struct tbvh_ctx_t* tbvh_ctx;   /* one per CUDA device */
typedef struct tbvh_bvh_t* tbvh_bvh;   /* one acceleration structure (any subset of the layouts) */
typedef struct tbvh_group_t* tbvh_group; /* several devices of one process: BVH replicas + index-sharded ray batches */

typedef struct tbvh_info
{
	uint32_t prim_count;     /* BVHBase::triCount */
	uint32_t idx_count;      /* BVHBase::idxCount */
	uint32_t used_nodes;     /* BVH::usedNodes (32-byte nodes, node 1 unused) */
	uint32_t used_nodes_gpu; /* BVH_GPU::usedNodes (64-byte nodes) */
	uint32_t used_blocks;    /* BVH8_CWBVH::usedBlocks (16-byte blocks; nodes = used_blocks/5) */
	uint32_t cwbvh_tri_count;/* BVH8_CWBVH triangle records (48 bytes each) */
	uint32_t max_depth;      /* depth of the BVH2 (root = 0) */
	uint32_t layouts;        /* bit (1<<TBVH_LAYOUT_*) per resident layout */
	float aabb_min[3], aabb_max[3]; /* BVHBase::aabbMin / aabbMax */
	double build_ms;         /* device time of the last tbvh_build on this handle */
} tbvh_info;

/* ---- context ---------------------------------------------------------------------------------------- */
int tbvh_ctx_create( int device, tbvh_ctx* out );
int tbvh_ctx_destroy( tbvh_ctx ctx );
const char* tbvh_last_error( void );
int tbvh_device_count( void );
/* host topology of a device: the NUMA node it hangs off (-1 when the system does not say), and a call that restricts the calling
 * thread (and the threads it creates afterwards) to that node's CPUs - ray buffers first-touched or page-locked from such a thread
 * are read by the device's DMA engine from local memory instead of across the socket interconnect. */
int tbvh_device_numa_node( int device );
int tbvh_bind_thread_to_device( int device );
/* context options (no reference counterpart).  Three keys; any other is TBVH_E_ARG:
 *  "inst_idx_bits"  the host program's INST_IDX_BITS, where a TLAS hit stores its instance (default 32, see tbvh_build_tlas)
 *  "small_t"        BVH::Build: subtrees of at most this many primitives are built by one warp each (8..128, default 128);
 *                   every value gives the same tree
 *  "build_mode"     BVH::Build large phase: 0 = one persistent cooperative launch (the default), 1 = one launch per stage and
 *                   level (what a device that refuses the cooperative launch runs); both give the same tree */
int tbvh_set_option( tbvh_ctx ctx, const char* key, int value );
/* pinned host memory for ray buffers (replaces tinybvh::malloc64 / BVHContext::malloc for rays, tiny_bvh.h:261-292, 763-768).
 * The pages are taken from the NUMA node of the current CUDA device (tbvh_host_alloc) or of `device` (_near); buffers of 8 MiB and more
 * are anonymous memory advised into transparent huge pages and then page-locked (TBVH_HOST_HUGE=0 switches that off): with an IOMMU
 * translating the DMA engine's addresses, 2 MiB pages are worth 5-9 % on the host-buffer path. */
int tbvh_host_alloc( size_t bytes, void** out );
int tbvh_host_alloc_near( int device, size_t bytes, void** out );
int tbvh_host_alloc_node( int numa_node, size_t bytes, void** out );
int tbvh_host_free( void* p );
int tbvh_host_register( void* p, size_t bytes );
int tbvh_host_unregister( void* p );

/* ---- acceleration structure --------------------------------------------------------------------------- */
int tbvh_bvh_create( tbvh_ctx ctx, tbvh_bvh* out );
int tbvh_bvh_destroy( tbvh_bvh bvh );
int tbvh_bvh_info( tbvh_bvh bvh, tbvh_info* out );

/* BVH::Build( const bvhvec4*, primCount ) tiny_bvh.h:2124 / Build( bvhvec4slice ) :2131 - binned SAH on the GPU.
 * verts: prim_count*3 vertices, `stride` bytes apart (16 for bvhvec4), xyz used.  The engine copies them
 * (the reference keeps a pointer: "we're not copying this data").  c_trav / c_int = BVHBase::c_trav, c_int. */
int tbvh_build( tbvh_bvh bvh, const void* verts, uint32_t stride, uint32_t prim_count, int space, float c_trav, float c_int );

/* The same builder with the decisions of BVH::BuildAVX (tiny_bvh.h:6400-6671) - the builder BuildDefault (:1817-1832) picks
 * on x86, i.e. what BVH_GPU::Build, BVH8_CWBVH::Build and BVH8_CPU::Build construct their trees with.  It differs from
 * BVH::Build in bin rounding, the partition's bin function, minDim and the plane tie-break order; the trees are
 * "nearly identical" (:6352) but not byte-identical, so both flavours exist. */
#define TBVH_BUILD_REFERENCE 0   /* BVH::Build */
#define TBVH_BUILD_AVX 1         /* BVH::BuildAVX / BuildDefault */
/* BVH::BuildHQ (tiny_bvh.h:2623-3040): SBVH - object split vs. spatial split with clipping (ClipFrag :8614, SplitFrag :8731)
 * and unsplitting, followed by Compact() (:3733).  idx_count becomes prim_count + prim_count/2 as in the reference (the
 * leaves reference the first sum(triCount) entries; the rest is zero), used_nodes up to 3 * prim_count. */
#define TBVH_BUILD_HQ 2          /* BVH::BuildHQ */
int tbvh_build_flavour( tbvh_bvh bvh, const void* verts, uint32_t stride, uint32_t prim_count, int space, float c_trav, float c_int, int flavour );

/* Indexed geometry: BVH::Build / BuildAVX / BuildHQ( const bvhvec4* vertices, const uint32_t* indices, primCount ) and their
 * bvhvec4slice forms (tiny_bvh.h:889-900; PrepareBuild reads verts[vertIdx[3 i + k]], :2290-2297).  verts: vert_count
 * vertices `stride` bytes apart; indices: 3 * prim_count entries.  primIdx numbers triangles exactly as the reference does
 * (triangle i = indices[3 i .. 3 i + 2]); an index >= vert_count is TBVH_E_ARG (the reference reads out of bounds). */
int tbvh_build_indexed( tbvh_bvh bvh, const void* verts, uint32_t stride, uint32_t vert_count, const uint32_t* indices, uint32_t prim_count, int space,
	float c_trav, float c_int, int flavour );

/* TLAS: BVH::Build( BLASInstance* instances, instCount, BVHBase** blasses, blasCount ) tiny_bvh.h:2221, traversed by
 * BVH::IntersectTLAS (:3306) / IsOccludedTLAS (:3455) whenever tbvh_intersect / tbvh_occluded (or the _device forms) are
 * called on the handle.  instances: inst_count records of the reference's 192-byte BLASInstance (:1443), inst_stride bytes
 * apart, ALREADY Update()d (invTransform and world box filled in: the reference's own "blasses == 0" mode, :2245);
 * blasses: handles holding a BVH-layout triangle tree in the same context - they must outlive the TLAS ("both must be kept
 * alive").  INST_IDX_BITS == 32 (the library default): a hit stores the instance number in hit.inst, byte 44 of the Ray
 * record, so closest hits are always returned in place (tbvh_intersect_packed / a separate d_hits array: TBVH_E_UNSUPPORTED).
 * A host program compiled with another INST_IDX_BITS (4..31) sets tbvh_set_option( ctx, "inst_idx_bits", bits ): hits then
 * carry the instance in the top bits of hit.prim (prim = triIdx + (inst << (32 - bits)), :8527) and byte 44 is left alone.
 * The `layout` argument of the traversal calls on a TLAS names the layout the BLASses are walked in: TBVH_LAYOUT_BVH (what the
 * reference's CPU IntersectTLAS does, :3341), or TBVH_LAYOUT_CWBVH - the arrangement of the reference's GPU path (traverse_tlas.cl:13-107:
 * BVH2 TLAS, per-instance ray transform, CWBVH BLASses, a BLAS hit kept when it is closer, the instance attached), semantics of
 * BVH8_CWBVH::Intersect (:7046) per BLAS.  A BLAS may hold either layout or both (CWBVH: tbvh_convert / tbvh_upload_cwbvh BEFORE
 * tbvh_build_tlas - the TLAS records the arrays each BLAS holds at that moment); walking a layout some BLAS did not hold is
 * TBVH_E_STATE, and so is walking a TLAS after one of its BLASses was rebuilt, re-converted, re-uploaded or destroyed. */
/* BVH::SAHCost( 0 ) tiny_bvh.h:1889-1897: the tree's SAH cost, host recursion over the (downloaded) 32-byte node array in the
 * reference's own order and rounding - the number the speedtest prints after every build.  _nodes works on a host array. */
int tbvh_sah_cost( tbvh_bvh bvh, float c_trav, float c_int, float* out );
int tbvh_sah_cost_nodes( const void* nodes32, uint32_t used_nodes, float c_trav, float c_int, float* out );

/* BLASInstance::Update( BVHBase* blas ) tiny_bvh.h:8386 on one 192-byte record: invTransform = inverse of transform
 * (InvertTransform :8402), aabbMin / aabbMax = box of the eight transformed corners of the BLAS's root box.  Host arithmetic in
 * the reference build's own operation order: the record comes out bit-identical to the reference's.  _box takes the root box
 * directly (no device needed). */
int tbvh_instance_update( void* instance, tbvh_bvh blas );
int tbvh_instance_update_box( void* instance, const float* blas_aabb_min, const float* blas_aabb_max );
int tbvh_build_tlas( tbvh_bvh tlas, const void* instances, uint32_t inst_stride, uint32_t inst_count, const tbvh_bvh* blasses, uint32_t blas_count,
	float c_trav, float c_int );

/* BVH::Refit (tiny_bvh.h:3055-3093): the triangles moved, the topology stays - leaf boxes from the new vertices, interior
 * boxes bottom-up.  verts as for tbvh_build, same prim_count.  TBVH_E_STATE for an SBVH (the reference's fatal "refitting an
 * SBVH") or when no BVH-layout tree is resident.  Derived layouts on the handle are dropped; tbvh_convert again. */
int tbvh_refit( tbvh_bvh bvh, const void* verts, uint32_t stride, uint32_t prim_count, int space );

/* consume a tree built elsewhere, in the reference's own layouts (the public members bvhNode / primIdx /
 * verts of tiny_bvh.h:952-964, BVH_GPU::bvhNode :1124, BVH8_CWBVH::bvh8Data / bvh8Tris :1356-1357) */
int tbvh_upload_bvh( tbvh_bvh bvh, const void* nodes32, uint32_t used_nodes, const uint32_t* prim_idx, uint32_t idx_count,
	const void* verts, uint32_t stride, uint32_t prim_count, int space );
int tbvh_upload_bvh_gpu( tbvh_bvh bvh, const void* nodes64, uint32_t used_nodes, const uint32_t* prim_idx, uint32_t idx_count,
	const void* verts, uint32_t stride, uint32_t prim_count, int space );
int tbvh_upload_cwbvh( tbvh_bvh bvh, const void* bvh8_data, uint32_t used_blocks, const void* bvh8_tris, uint32_t tri_count, int space );

/* layout conversion on the device: BVH_GPU::ConvertFrom tiny_bvh.h:4612; BVH8_CWBVH::Build's chain
 * Compact :3733 + SplitLeafs(3) :1988 + MBVH<8>::ConvertFrom :4975 + BVH8_CWBVH::ConvertFrom :5884 */
int tbvh_convert( tbvh_bvh bvh, int to_layout );

/* read a layout back in the reference's format so SAHCost / Save / ConvertFrom / the CPU traversals can use a
 * GPU-built tree.  Buffers are sized from tbvh_bvh_info. */
int tbvh_download_bvh( tbvh_bvh bvh, void* nodes32, uint32_t* prim_idx, int space );
int tbvh_download_bvh_gpu( tbvh_bvh bvh, void* nodes64, int space );
int tbvh_download_cwbvh( tbvh_bvh bvh, void* bvh8_data, void* bvh8_tris, int space );

/* ---- traversal ------------------------------------------------------------------------------------------ */
/* BVH::Intersect( Ray& ) tiny_bvh.h:3222 / BVH_GPU::Intersect :4657 / BVH8_CWBVH::Intersect :7046 and the OpenCL
 * batch kernels batch_ailalaine (traverse_bvh2.cl:209) / batch_cwbvh (traverse_cwbvh.cl:554) for a whole batch:
 * host records, in place - copies bytes 0..63 in, writes t,u,v,prim back to bytes 48..63 of every record. */
int tbvh_intersect( tbvh_bvh bvh, int layout, void* rays, uint32_t stride, uint64_t n );
/* same traversal, hits delivered as a packed array of 16-byte (t,u,v,prim) records instead of being scattered into the
 * 128-byte ray records: the return trip becomes one contiguous copy per chunk (the in-place form returns bytes 0..63
 * of every record in a strided copy; see DESIGN.md 4.5).  `rays` is not modified. */
int tbvh_intersect_packed( tbvh_bvh bvh, int layout, const void* rays, uint32_t stride, uint64_t n, void* hits );
/* BVH::IsOccluded( const Ray& ) tiny_bvh.h:3382 / isoccluded_cwbvh (traverse_cwbvh.cl:343) for a batch:
 * bits[i>>5] bit (i&31) = occluded; (n+31)/32 words are written. */
int tbvh_occluded( tbvh_bvh bvh, int layout, const void* rays, uint32_t stride, uint64_t n, uint32_t* bits );

/* the same with everything already resident in HBM, asynchronous on `stream` (a cudaStream_t, 0 = default).
 * hits == NULL writes t,u,v,prim into bytes 48..63 of each record; otherwise 16-byte records to hits[]. */
int tbvh_intersect_device( tbvh_bvh bvh, int layout, void* d_rays, uint32_t stride, void* d_hits, uint64_t n, void* stream );
int tbvh_occluded_device( tbvh_bvh bvh, int layout, const void* d_rays, uint32_t stride, uint32_t* d_bits, uint64_t n, void* stream );

/* counters of the last device traversal on this handle when statistics are enabled (debug aid; the reference
 * returns the per-ray cost from Intersect, tiny_bvh.h:3303): steps = nodes visited, tris = triangle tests. */
int tbvh_set_stats( tbvh_bvh bvh, int enable );
int tbvh_get_stats( tbvh_bvh bvh, uint64_t* steps, uint64_t* tris );
/* the same plus the CWBVH kernels' child-pair steps: out = { node visits, triangle tests, pair steps, 0 } */
int tbvh_get_stats_ex( tbvh_bvh bvh, uint64_t out[4] );
/* rays[0..n) of a host buffer -> packed 64-byte device records (bytes 0..63 of each record; the speedtest's upload,
 * tiny_bvh_speedtest.cpp:1110-1115), asynchronous on `stream` */
int tbvh_copy_rays_to_device( const void* rays, uint32_t stride, uint64_t n, void* d_rays, void* stream );
/* device memory / synchronisation for host programs that do not link the CUDA runtime themselves (the role tinyocl::Buffer plays
 * in the reference's GPU section, tiny_bvh_speedtest.cpp:1100-1115): cudaMalloc / cudaFree / cudaDeviceSynchronize / a blocking
 * device-to-host copy on the context's device */
int tbvh_device_alloc( tbvh_ctx ctx, size_t bytes, void** out );
int tbvh_device_free( tbvh_ctx ctx, void* p );
int tbvh_device_sync( tbvh_ctx ctx );
int tbvh_copy_from_device( void* host, const void* d_src, size_t bytes );

/* ---- several GPUs in one process (SURVEY.md 8(e): rays shard by index, the BVH is replicated once, no traffic between devices
 * during traversal).  The reference has no counterpart: its GPU path drives one OpenCL device (tiny_bvh_speedtest.cpp:1092-1241).
 *  tbvh_group_create     devices[count] (NULL / 0 = all devices), one engine context each, peer access enabled where possible
 *  tbvh_group_replicate  copy the traversal arrays of a built / uploaded / converted BVH to every device of the group (peer copies
 *                        over NVLink); ms_out = device time of the copies.  Call again after the source changed.
 *  tbvh_group_intersect / _occluded  tbvh_intersect / tbvh_occluded on a HOST batch, rays [first, first+count) of
 *                        tbvh_shard_range( n, g, size ) going to device g from a worker thread bound to that device's NUMA node
 *  tbvh_group_host_alloc page-locked buffer of n records whose index ranges live on the NUMA node of the device that reads them
 *  tbvh_shard_range      the partition itself: contiguous, boundaries on multiples of 32 rays (occlusion words are never shared) */
int tbvh_group_create( const int* devices, int count, tbvh_group* out );
int tbvh_group_destroy( tbvh_group group );
int tbvh_group_size( tbvh_group group );
tbvh_ctx tbvh_group_ctx( tbvh_group group, int i );
tbvh_bvh tbvh_group_replica( tbvh_group group, int i );
int tbvh_group_replicate( tbvh_group group, tbvh_bvh src, double* ms_out );
int tbvh_group_intersect( tbvh_group group, int layout, void* rays, uint32_t stride, uint64_t n );
int tbvh_group_occluded( tbvh_group group, int layout, const void* rays, uint32_t stride, uint64_t n, uint32_t* bits );
int tbvh_group_host_alloc( tbvh_group group, uint32_t stride, uint64_t n, void** out );
int tbvh_group_host_free( tbvh_group group, void* p );
void tbvh_shard_range( uint64_t n, uint32_t part, uint32_t parts, uint64_t* first, uint64_t* count );

/* number of kernels this library has launched since load (bench.py reports it as gpu_launches) */
uint64_t tbvh_launch_count( void );

#ifdef __cplusplus
}
#endif
#endif
