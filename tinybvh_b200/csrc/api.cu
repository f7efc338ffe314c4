// tinybvh_b200/csrc/api.cu - C-ABI entry points (include/tinybvh_b200.h): contexts, handles, uploads, the host-buffer
// traversal pipeline.  Kernels live in trace_bvh2.cu / trace_cwbvh.cu / build_sah.cu / convert.cu.
#include "common.cuh"
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <mutex>
#include <new>

static thread_local char g_err[512] = "";
unsigned long long g_tbvh_launches = 0;

void tbvh_set_error( const char* fmt, ... )
{
	va_list ap;
	va_start( ap, fmt );
	vsnprintf( g_err, sizeof( g_err ), fmt, ap );
	va_end( ap );
}

#define ARG_CHECK( c, msg ) do { if (!(c)) { tbvh_set_error( "%s: %s", __func__, msg ); return TBVH_E_ARG; } } while (0)
#define TRY( x ) do { int r_ = (x); if (r_ != TBVH_OK) return r_; } while (0)


// ---- host topology: which NUMA node a device hangs off, and its CPUs (sysfs; no libnuma in the image) -----------------
#include <sched.h>
#include <unistd.h>
#include <sys/mman.h>
#include <sys/syscall.h>

static int read_int_file( const char* path, int fallback )
{
	FILE* f = fopen( path, "r" );
	if (!f) return fallback;
	int v = fallback;
	if (fscanf( f, "%d", &v ) != 1) v = fallback;
	fclose( f );
	return v;
}

static int device_numa_node( int device )
{
	char bus[32] = "";
	if (cudaDeviceGetPCIBusId( bus, sizeof( bus ), device ) != cudaSuccess) { cudaGetLastError(); return -1; }
	for (char* c = bus; *c; c++) if (*c >= 'A' && *c <= 'Z') *c += 'a' - 'A';
	char path[128];
	snprintf( path, sizeof( path ), "/sys/bus/pci/devices/%s/numa_node", bus );
	return read_int_file( path, -1 );
}

// CPUs of a NUMA node from /sys/devices/system/node/nodeN/cpulist ("0-31,64-95")
static bool node_cpus( int node, cpu_set_t* set )
{
	CPU_ZERO( set );
	if (node < 0) return false;
	char path[128], line[1024] = "";
	snprintf( path, sizeof( path ), "/sys/devices/system/node/node%d/cpulist", node );
	FILE* f = fopen( path, "r" );
	if (!f) return false;
	const bool ok = fgets( line, sizeof( line ), f ) != 0;
	fclose( f );
	if (!ok) return false;
	int any = 0;
	for (char* p = line; *p && *p != '\n';)
	{
		char* e;
		long lo = strtol( p, &e, 10 ), hi = lo;
		if (e == p) break;
		if (*e == '-') { p = e + 1; hi = strtol( p, &e, 10 ); }
		for (long c = lo; c <= hi && c < CPU_SETSIZE; c++) CPU_SET( (int)c, set ), any = 1;
		p = *e == ',' ? e + 1 : e;
	}
	return any != 0;
}

// run `fn` with the calling thread restricted to the CPUs of `node` (first-touch and driver allocations then land on that node),
// then restore the previous affinity.  Without topology information fn just runs.
template <class F> static auto on_node( int node, F fn ) -> decltype( fn() )
{
	cpu_set_t want, old;
	const bool have = node_cpus( node, &want ) && sched_getaffinity( 0, sizeof( old ), &old ) == 0 && sched_setaffinity( 0, sizeof( want ), &want ) == 0;
	auto r = fn();
	if (have) sched_setaffinity( 0, sizeof( old ), &old );
	return r;
}

extern "C" {

const char* tbvh_last_error( void ) { return g_err; }
uint64_t tbvh_launch_count( void ) { return g_tbvh_launches; }

int tbvh_device_count( void )
{
	int n = 0;
	if (cudaGetDeviceCount( &n ) != cudaSuccess) { cudaGetLastError(); return 0; }
	return n;
}

int tbvh_device_numa_node( int device ) { return device_numa_node( device ); }

int tbvh_bind_thread_to_device( int device )
{
	cpu_set_t want;
	const int node = device_numa_node( device );
	if (!node_cpus( node, &want )) { tbvh_set_error( "tbvh_bind_thread_to_device: no NUMA information for device %d", device ); return TBVH_E_UNSUPPORTED; }
	if (sched_setaffinity( 0, sizeof( want ), &want ) != 0) { tbvh_set_error( "tbvh_bind_thread_to_device: sched_setaffinity failed" ); return TBVH_E_UNSUPPORTED; }
	return TBVH_OK;
}

int tbvh_ctx_destroy( tbvh_ctx c );

int tbvh_ctx_create( int device, tbvh_ctx* out )
{
	ARG_CHECK( out, "out == NULL" );
	int n = 0;
	CUDA_TRY( cudaGetDeviceCount( &n ) );
	if (device < 0 || device >= n) { tbvh_set_error( "tbvh_ctx_create: device %d of %d - no CUDA device, and there is no CPU fallback", device, n ); return TBVH_E_CUDA; }
	CUDA_TRY( cudaSetDevice( device ) );
	tbvh_ctx c = new (std::nothrow) tbvh_ctx_t();
	ARG_CHECK( c, "out of host memory" );
	c->device = device;
	auto body = [&]() -> int
	{
		cudaDeviceProp prop;
		CUDA_TRY( cudaGetDeviceProperties( &prop, device ) );
		c->sm_count = prop.multiProcessorCount;
		CUDA_TRY( cudaStreamCreateWithFlags( &c->stream, cudaStreamNonBlocking ) );
		CUDA_TRY( cudaStreamCreateWithFlags( &c->s_in, cudaStreamNonBlocking ) );
		CUDA_TRY( cudaStreamCreateWithFlags( &c->s_run, cudaStreamNonBlocking ) );
		CUDA_TRY( cudaStreamCreateWithFlags( &c->s_out, cudaStreamNonBlocking ) );
		for (int i = 0; i < TBVH_SLOTS; i++)
		{
			CUDA_TRY( cudaEventCreateWithFlags( &c->slot[i].in_done, cudaEventDisableTiming ) );
			CUDA_TRY( cudaEventCreateWithFlags( &c->slot[i].run_done, cudaEventDisableTiming ) );
			CUDA_TRY( cudaEventCreateWithFlags( &c->slot[i].out_done, cudaEventDisableTiming ) );
		}
		return TBVH_OK;
	};
	const int rc = body();
	if (rc != TBVH_OK) { tbvh_ctx_destroy( c ); return rc; }
	*out = c;
	return TBVH_OK;
}

int tbvh_ctx_destroy( tbvh_ctx c )
{
	if (!c) return TBVH_OK;
	cudaSetDevice( c->device );
	cudaDeviceSynchronize();
	for (int i = 0; i < TBVH_SLOTS; i++)
	{
		if (c->slot[i].d_rays) cudaFree( c->slot[i].d_rays );
		if (c->slot[i].d_hits) cudaFree( c->slot[i].d_hits );
		if (c->slot[i].d_bits) cudaFree( c->slot[i].d_bits );
		if (c->slot[i].in_done) cudaEventDestroy( c->slot[i].in_done );
		if (c->slot[i].run_done) cudaEventDestroy( c->slot[i].run_done );
		if (c->slot[i].out_done) cudaEventDestroy( c->slot[i].out_done );
	}
	if (c->s_in) cudaStreamDestroy( c->s_in );
	if (c->s_run) cudaStreamDestroy( c->s_run );
	if (c->s_out) cudaStreamDestroy( c->s_out );
	if (c->stream) cudaStreamDestroy( c->stream );
	delete c;
	return TBVH_OK;
}

int tbvh_set_option( tbvh_ctx c, const char* key, int value )
{
	ARG_CHECK( c && key, "NULL argument" );
	if (!strcmp( key, "inst_idx_bits" )) c->inst_idx_bits = value;
	else if (!strcmp( key, "small_t" )) c->small_t = value;
	else if (!strcmp( key, "build_mode" )) c->build_mode = value ? 1 : 0;
	else { tbvh_set_error( "tbvh_set_option: unknown key '%s'", key ); return TBVH_E_ARG; }
	return TBVH_OK;
}

// Page-locked ray buffers.  The pages are allocated while the calling thread sits on the CPUs of the device's NUMA node, so the
// DMA engine reads local memory (a dual-socket host serves a remote GPU's reads over the inter-socket link otherwise).
// blocks handed out by the huge-page path (mmap + MADV_HUGEPAGE + cudaHostRegister): tbvh_host_free must munmap them
static std::mutex g_huge_mutex;
static std::vector<std::pair<void*, size_t>> g_huge;

static int host_alloc_on_node( int node, size_t bytes, void** out );
int tbvh_host_alloc_near( int device, size_t bytes, void** out ) { return host_alloc_on_node( device_numa_node( device ), bytes, out ); }
int tbvh_host_alloc_node( int node, size_t bytes, void** out ) { return host_alloc_on_node( node, bytes, out ); }
static int host_alloc_on_node( int node, size_t bytes, void** out )
{
	ARG_CHECK( out, "out == NULL" );
	static int huge = -1;
	if (huge < 0) { const char* e = getenv( "TBVH_HOST_HUGE" ); huge = e ? atoi( e ) : 1; } // default on: +5..9 % on the host path where the IOMMU translates DMA addresses (profiles/README.md)
	if (huge && bytes >= (8u << 20))
	{
		// anonymous memory advised into transparent huge pages, first touched on the device's node, then page-locked: 2 MiB pages
		// mean 512x fewer IOMMU / address-translation entries for the DMA engine than 4 KiB ones
		const size_t sz = (bytes + (2u << 20) - 1) & ~(size_t)((2u << 20) - 1);
		void* p = mmap( 0, sz, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0 );
		if (p != MAP_FAILED)
		{
			madvise( p, sz, MADV_HUGEPAGE );
			const cudaError_t e = on_node( node, [&]() { for (size_t o = 0; o < sz; o += 4096) ((volatile char*)p)[o] = 0; return cudaHostRegister( p, sz, cudaHostRegisterPortable ); } );
			if (e == cudaSuccess) { std::lock_guard<std::mutex> lk( g_huge_mutex ); g_huge.push_back( { p, sz } ); *out = p; return TBVH_OK; }
			cudaGetLastError();
			munmap( p, sz );
		}
	}
	const cudaError_t e = on_node( node, [&]() { return cudaHostAlloc( out, bytes, cudaHostAllocPortable ); } );
	if (e != cudaSuccess) { tbvh_set_error( "tbvh_host_alloc: cudaHostAlloc( %zu ) -> %s", bytes, cudaGetErrorString( e ) ); return TBVH_E_CUDA; }
	return TBVH_OK;
}
int tbvh_host_alloc( size_t bytes, void** out )
{
	int device = 0;
	if (cudaGetDevice( &device ) != cudaSuccess) { cudaGetLastError(); device = 0; }
	return tbvh_host_alloc_near( device, bytes, out );
}
int tbvh_host_free( void* p )
{
	if (!p) return TBVH_OK;
	{
		std::lock_guard<std::mutex> lk( g_huge_mutex );
		for (size_t i = 0; i < g_huge.size(); i++) if (g_huge[i].first == p)
		{
			cudaHostUnregister( p );
			munmap( p, g_huge[i].second );
			g_huge.erase( g_huge.begin() + i );
			return TBVH_OK;
		}
	}
	CUDA_TRY( cudaFreeHost( p ) );
	return TBVH_OK;
}
int tbvh_host_register( void* p, size_t bytes ) { CUDA_TRY( cudaHostRegister( p, bytes, cudaHostRegisterPortable ) ); return TBVH_OK; }
int tbvh_host_unregister( void* p ) { CUDA_TRY( cudaHostUnregister( p ) ); return TBVH_OK; }

static void live_add( tbvh_bvh b );
static void live_remove( tbvh_bvh b );

int tbvh_bvh_create( tbvh_ctx ctx, tbvh_bvh* out )
{
	ARG_CHECK( ctx && out, "NULL argument" );
	tbvh_bvh b = new (std::nothrow) tbvh_bvh_t();
	ARG_CHECK( b, "out of host memory" );
	b->ctx = ctx;
	const cudaError_t ce = cudaSetDevice( ctx->device ) != cudaSuccess ? cudaGetLastError() : cudaMalloc( &b->d_stats, 32 );
	if (ce != cudaSuccess || cudaMemset( b->d_stats, 0, 32 ) != cudaSuccess)
	{
		tbvh_set_error( "tbvh_bvh_create: %s", cudaGetErrorString( ce != cudaSuccess ? ce : cudaGetLastError() ) );
		if (b->d_stats) cudaFree( b->d_stats );
		delete b;
		return TBVH_E_CUDA;
	}
	b->generation = tbvh_next_generation();
	live_add( b );
	*out = b;
	return TBVH_OK;
}

static void free_layouts( tbvh_bvh b )
{
	if (b->d_trav && b->d_trav != b->d_nodes) cudaFree( b->d_trav );
	void* p[] = { b->d_verts, b->d_nodes, b->d_prim_idx, b->d_leaf_tris, b->d_nodes_gpu, b->d_cw_nodes, b->d_cw_tris, b->d_cw_trav, b->d_aabbs, b->d_inst, b->d_blas };
	for (void* q : p) if (q) cudaFree( q );
	b->d_verts = 0, b->d_nodes = 0, b->d_prim_idx = 0, b->d_leaf_tris = 0, b->d_nodes_gpu = 0, b->d_cw_nodes = 0, b->d_cw_tris = 0, b->d_cw_trav = 0, b->d_trav = 0, b->leaf_tris_count = 0;
	b->d_aabbs = 0, b->d_inst = 0, b->d_blas = 0, b->inst_count = 0, b->blas_count = 0, b->cw_depth = 0, b->tlas_blas_layouts = 0;
	b->links.clear();
	b->generation = tbvh_next_generation(); // a TLAS built over the old arrays must notice (tlas_check)
	memset( &b->info, 0, sizeof( b->info ) );
	b->refittable = true;
}

int tbvh_bvh_destroy( tbvh_bvh b )
{
	if (!b) return TBVH_OK;
	cudaSetDevice( b->ctx->device );
	live_remove( b );
	free_layouts( b );
	if (b->d_stats) cudaFree( b->d_stats );
	delete b;
	return TBVH_OK;
}

int tbvh_bvh_info( tbvh_bvh b, tbvh_info* out ) { ARG_CHECK( b && out, "NULL argument" ); *out = b->info; return TBVH_OK; }
int tbvh_set_stats( tbvh_bvh b, int enable ) { ARG_CHECK( b, "NULL handle" ); b->stats = enable; return TBVH_OK; }
int tbvh_get_stats( tbvh_bvh b, uint64_t* steps, uint64_t* tris )
{
	ARG_CHECK( b, "NULL handle" );
	unsigned long long h[2];
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	CUDA_TRY( cudaDeviceSynchronize() );
	CUDA_TRY( cudaMemcpy( h, b->d_stats, 16, cudaMemcpyDeviceToHost ) );
	if (steps) *steps = h[0];
	if (tris) *tris = h[1];
	return TBVH_OK;
}
int tbvh_get_stats_ex( tbvh_bvh b, uint64_t out[4] )
{
	ARG_CHECK( b && out, "NULL argument" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	CUDA_TRY( cudaDeviceSynchronize() );
	CUDA_TRY( cudaMemcpy( out, b->d_stats, 32, cudaMemcpyDeviceToHost ) );
	return TBVH_OK;
}

} // extern "C"

// ---- uploads ------------------------------------------------------------------------------------------------

// vertices -> engine-owned float4 array (xyz of each vertex, w copied when the stride holds it)
static int upload_verts( tbvh_bvh b, const void* verts, uint32_t stride, uint32_t prim_count, int space, cudaStream_t s )
{
	ARG_CHECK( verts && stride >= 12 && (stride & 3) == 0 && prim_count > 0, "bad vertex slice" );
	const size_t nv = (size_t)prim_count * 3;
	CUDA_TRY( cudaMalloc( &b->d_verts, nv * 16 ) );
	const cudaMemcpyKind kind = space == TBVH_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	if (stride == 16) CUDA_TRY( cudaMemcpyAsync( b->d_verts, verts, nv * 16, kind, s ) );
	else
	{
		CUDA_TRY( cudaMemsetAsync( b->d_verts, 0, nv * 16, s ) );
		CUDA_TRY( cudaMemcpy2DAsync( b->d_verts, 16, verts, stride, stride < 16 ? stride : 16, nv, kind, s ) );
	}
	b->info.prim_count = prim_count;
	return TBVH_OK;
}

// indexed geometry (the `vertices, indices, primCount` overloads, tiny_bvh.h:889-900): the engine keeps its own copy of
// the vertices anyway, so the indices are resolved once, on the device, into the flat 3-vertices-per-triangle array the
// kernels read.  The tree is the one the reference builds with vertIdx set (same fragments, same primIdx numbering).
__global__ void k_gather_verts( const float4* __restrict__ src, const uint32_t* __restrict__ indices, float4* __restrict__ dst, const uint32_t n, const uint32_t vert_count, uint32_t* bad )
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const uint32_t v = indices[i];
	if (v >= vert_count) { atomicAdd( bad, 1u ); dst[i] = make_float4( 0, 0, 0, 0 ); return; }
	dst[i] = src[v];
}
static int upload_verts_indexed( tbvh_bvh b, const void* verts, uint32_t stride, uint32_t vert_count, const uint32_t* indices, uint32_t prim_count, int space, cudaStream_t s )
{
	ARG_CHECK( verts && indices && stride >= 12 && (stride & 3) == 0 && prim_count > 0 && vert_count > 0, "bad indexed vertex slice" );
	const size_t nv = (size_t)prim_count * 3;
	const cudaMemcpyKind kind = space == TBVH_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	float4* d_src = 0; uint32_t* d_idx = 0; uint32_t* d_bad = 0;
	int rc = TBVH_OK;
	auto body = [&]() -> int
	{
		CUDA_TRY( cudaMalloc( &d_src, (size_t)vert_count * 16 ) );
		CUDA_TRY( cudaMalloc( &d_idx, nv * 4 ) );
		CUDA_TRY( cudaMalloc( &d_bad, 4 ) );
		CUDA_TRY( cudaMalloc( &b->d_verts, nv * 16 ) );
		CUDA_TRY( cudaMemsetAsync( d_bad, 0, 4, s ) );
		if (stride == 16) CUDA_TRY( cudaMemcpyAsync( d_src, verts, (size_t)vert_count * 16, kind, s ) );
		else
		{
			CUDA_TRY( cudaMemsetAsync( d_src, 0, (size_t)vert_count * 16, s ) );
			CUDA_TRY( cudaMemcpy2DAsync( d_src, 16, verts, stride, stride < 16 ? stride : 16, vert_count, kind, s ) );
		}
		CUDA_TRY( cudaMemcpyAsync( d_idx, indices, nv * 4, kind, s ) );
		k_gather_verts<<<(unsigned)((nv + 255) / 256), 256, 0, s>>>( d_src, d_idx, b->d_verts, (uint32_t)nv, vert_count, d_bad ); LAUNCHED();
		uint32_t bad = 0;
		CUDA_TRY( cudaMemcpyAsync( &bad, d_bad, 4, cudaMemcpyDeviceToHost, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		if (bad) { tbvh_set_error( "indexed build: %u indices point past the %u vertices", bad, vert_count ); return TBVH_E_ARG; }
		return TBVH_OK;
	};
	rc = body();
	cudaFree( d_src ), cudaFree( d_idx ), cudaFree( d_bad );
	b->info.prim_count = prim_count;
	return rc;
}

static uint32_t depth_of_bvh( const uint32_t* nodes /* 8 words per node */, uint32_t used_nodes )
{
	// iterative DFS over Wald nodes; returns the depth of the deepest node (root = 0)
	std::vector<uint2> st;
	st.push_back( make_uint2( 0, 0 ) );
	uint32_t maxd = 0;
	while (!st.empty())
	{
		const uint2 e = st.back();
		st.pop_back();
		if (e.y > maxd) maxd = e.y;
		const uint32_t* n = nodes + (size_t)e.x * 8;
		if (n[7] == 0 && n[3] + 1 < used_nodes) { st.push_back( make_uint2( n[3], e.y + 1 ) ); st.push_back( make_uint2( n[3] + 1, e.y + 1 ) ); }
	}
	return maxd;
}

static uint32_t depth_of_bvh_gpu( const uint32_t* nodes /* 16 words per node */, uint32_t used_nodes )
{
	std::vector<uint2> st;
	st.push_back( make_uint2( 0, 0 ) );
	uint32_t maxd = 0;
	while (!st.empty())
	{
		const uint2 e = st.back();
		st.pop_back();
		if (e.y > maxd) maxd = e.y;
		const uint32_t* n = nodes + (size_t)e.x * 16;
		if (n[11] == 0 && n[3] < used_nodes && n[7] < used_nodes) { st.push_back( make_uint2( n[3], e.y + 1 ) ); st.push_back( make_uint2( n[7], e.y + 1 ) ); }
	}
	return maxd;
}

extern "C" {

int tbvh_upload_bvh( tbvh_bvh b, const void* nodes32, uint32_t used_nodes, const uint32_t* prim_idx, uint32_t idx_count,
	const void* verts, uint32_t stride, uint32_t prim_count, int space )
{
	ARG_CHECK( b && nodes32 && prim_idx && used_nodes >= 1 && idx_count >= 1, "bad tree arrays" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	cudaStream_t s = b->ctx->stream;
	free_layouts( b );
	TRY( upload_verts( b, verts, stride, prim_count, space, s ) );
	const cudaMemcpyKind kind = space == TBVH_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	CUDA_TRY( cudaMalloc( &b->d_nodes, (size_t)(used_nodes < 2 ? 2 : used_nodes) * 32 ) );
	CUDA_TRY( cudaMemcpyAsync( b->d_nodes, nodes32, (size_t)used_nodes * 32, kind, s ) );
	CUDA_TRY( cudaMalloc( &b->d_prim_idx, (size_t)idx_count * 4 ) );
	CUDA_TRY( cudaMemcpyAsync( b->d_prim_idx, prim_idx, (size_t)idx_count * 4, kind, s ) );
	// root record + depth from a host copy of the nodes
	std::vector<uint32_t> host;
	const uint32_t* hn = (const uint32_t*)nodes32;
	if (space == TBVH_DEVICE)
	{
		host.resize( (size_t)used_nodes * 8 );
		CUDA_TRY( cudaMemcpyAsync( host.data(), nodes32, (size_t)used_nodes * 32, cudaMemcpyDeviceToHost, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		hn = host.data();
	}
	b->root_ref = hn[3], b->root_count = hn[7];
	b->info.used_nodes = used_nodes, b->info.idx_count = idx_count;
	b->info.max_depth = depth_of_bvh( hn, used_nodes );
	memcpy( b->info.aabb_min, hn, 12 ), memcpy( b->info.aabb_max, hn + 4, 12 );
	b->d_trav = b->d_nodes;
	TRY( make_leaf_tris( b, s ) );
	CUDA_TRY( cudaStreamSynchronize( s ) );
	b->info.layouts = 1u << TBVH_LAYOUT_BVH;
	return TBVH_OK;
}

int tbvh_upload_bvh_gpu( tbvh_bvh b, const void* nodes64, uint32_t used_nodes, const uint32_t* prim_idx, uint32_t idx_count,
	const void* verts, uint32_t stride, uint32_t prim_count, int space )
{
	ARG_CHECK( b && nodes64 && prim_idx && used_nodes >= 1 && idx_count >= 1, "bad tree arrays" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	cudaStream_t s = b->ctx->stream;
	free_layouts( b );
	TRY( upload_verts( b, verts, stride, prim_count, space, s ) );
	const cudaMemcpyKind kind = space == TBVH_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	CUDA_TRY( cudaMalloc( &b->d_nodes_gpu, (size_t)used_nodes * 64 ) );
	CUDA_TRY( cudaMemcpyAsync( b->d_nodes_gpu, nodes64, (size_t)used_nodes * 64, kind, s ) );
	CUDA_TRY( cudaMalloc( &b->d_prim_idx, (size_t)idx_count * 4 ) );
	CUDA_TRY( cudaMemcpyAsync( b->d_prim_idx, prim_idx, (size_t)idx_count * 4, kind, s ) );
	std::vector<uint32_t> host;
	const uint32_t* hn = (const uint32_t*)nodes64;
	if (space == TBVH_DEVICE)
	{
		host.resize( (size_t)used_nodes * 16 );
		CUDA_TRY( cudaMemcpyAsync( host.data(), nodes64, (size_t)used_nodes * 64, cudaMemcpyDeviceToHost, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		hn = host.data();
	}
	b->info.used_nodes_gpu = used_nodes, b->info.idx_count = idx_count;
	b->info.max_depth = depth_of_bvh_gpu( hn, used_nodes );
	// root as a child record: a leaf root keeps (firstTri, triCount); an interior root is pair 0 (pairs are indexed by 2*node)
	if (hn[11] > 0) b->root_ref = hn[15], b->root_count = hn[11]; else b->root_ref = 0, b->root_count = 0;
	TRY( bvh_gpu_to_bvh( b, used_nodes, s ) );
	TRY( make_leaf_tris( b, s ) );
	CUDA_TRY( cudaStreamSynchronize( s ) );
	b->info.layouts = 1u << TBVH_LAYOUT_BVH_GPU;
	return TBVH_OK;
}

int tbvh_upload_cwbvh( tbvh_bvh b, const void* bvh8_data, uint32_t used_blocks, const void* bvh8_tris, uint32_t tri_count, int space )
{
	ARG_CHECK( b && bvh8_data && bvh8_tris && used_blocks >= 5 && tri_count >= 1, "bad CWBVH arrays" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	cudaStream_t s = b->ctx->stream;
	const cudaMemcpyKind kind = space == TBVH_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	ARG_CHECK( used_blocks % 5 == 0, "usedBlocks must be a multiple of 5 (80-byte nodes)" );
	if (b->d_cw_trav || b->d_cw_tris) b->generation = tbvh_next_generation(); // a TLAS may hold these addresses (tlas_check)
	if (b->d_cw_nodes) cudaFree( b->d_cw_nodes );
	if (b->d_cw_tris) cudaFree( b->d_cw_tris );
	if (b->d_cw_trav) cudaFree( b->d_cw_trav );
	b->d_cw_nodes = 0, b->d_cw_tris = 0, b->d_cw_trav = 0;
	CUDA_TRY( cudaMalloc( &b->d_cw_nodes, (size_t)used_blocks * 16 ) );
	CUDA_TRY( cudaMalloc( &b->d_cw_tris, (size_t)tri_count * 48 ) );
	CUDA_TRY( cudaMemcpyAsync( b->d_cw_nodes, bvh8_data, (size_t)used_blocks * 16, kind, s ) );
	CUDA_TRY( cudaMemcpyAsync( b->d_cw_tris, bvh8_tris, (size_t)tri_count * 48, kind, s ) );
	b->info.used_blocks = used_blocks, b->info.cwbvh_tri_count = tri_count;
	TRY( cw_make_trav( b, s ) ); // the traversal nodes the kernels read + the wide tree's depth (synchronises the stream)
	b->info.layouts |= 1u << TBVH_LAYOUT_CWBVH;
	return TBVH_OK;
}

int tbvh_build_flavour( tbvh_bvh b, const void* verts, uint32_t stride, uint32_t prim_count, int space, float c_trav, float c_int, int flavour )
{
	ARG_CHECK( b, "NULL handle" );
	ARG_CHECK( flavour == TBVH_BUILD_REFERENCE || flavour == TBVH_BUILD_AVX || flavour == TBVH_BUILD_HQ, "unknown builder flavour" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	free_layouts( b );
	TRY( upload_verts( b, verts, stride, prim_count, space, b->ctx->stream ) );
	if (flavour == TBVH_BUILD_HQ) TRY( build_hq_launch( b, c_trav, c_int ) ); else TRY( build_sah_launch( b, c_trav, c_int, flavour ) );
	b->info.layouts = 1u << TBVH_LAYOUT_BVH, b->refittable = flavour != TBVH_BUILD_HQ;
	return TBVH_OK;
}

// ---- BVH::SAHCost (tiny_bvh.h:1889-1897) over a downloaded node array: host recursion in the reference's own order
__attribute__( (optimize( "fp-contract=off" )) ) static float sah_rec( const float* nodes /* 8 words per node */, const uint32_t i, const float c_trav, const float c_int )
{
	const float* n = nodes + (size_t)i * 8;
	uint32_t leftFirst, triCount;
	memcpy( &leftFirst, n + 3, 4 ), memcpy( &triCount, n + 7, 4 );
	const float ex = n[4] - n[0], ey = n[5] - n[1], ez = n[6] - n[2];
	const float sa = fmaf( ez, ex, fmaf( ey, ex, ey * ez ) ); // BVHBase::SA :8477 in the reference build's pairing
	if (triCount > 0) return c_int * sa * triCount;
	return c_trav * sa + sah_rec( nodes, leftFirst, c_trav, c_int ) + sah_rec( nodes, leftFirst + 1, c_trav, c_int );
}
__attribute__( (optimize( "fp-contract=off" )) ) int tbvh_sah_cost_nodes( const void* nodes32, uint32_t used_nodes, float c_trav, float c_int, float* out )
{
	ARG_CHECK( nodes32 && used_nodes >= 1 && out, "bad arguments" );
	const float* n = (const float*)nodes32;
	const float cost = sah_rec( n, 0, c_trav, c_int );
	const float ex = n[4] - n[0], ey = n[5] - n[1], ez = n[6] - n[2];
	*out = cost / fmaf( ez, ex, fmaf( ey, ex, ey * ez ) ); // the root divides by its own area (:1896)
	return TBVH_OK;
}
int tbvh_sah_cost( tbvh_bvh b, float c_trav, float c_int, float* out )
{
	ARG_CHECK( b && out, "NULL argument" );
	if (!(b->info.layouts & (1u << TBVH_LAYOUT_BVH)) || !b->d_nodes) { tbvh_set_error( "tbvh_sah_cost: no BVH-layout tree on this handle" ); return TBVH_E_STATE; }
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	std::vector<float> nodes( (size_t)b->info.used_nodes * 8 );
	CUDA_TRY( cudaMemcpy( nodes.data(), b->d_nodes, nodes.size() * 4, cudaMemcpyDeviceToHost ) );
	return tbvh_sah_cost_nodes( nodes.data(), b->info.used_nodes, c_trav, c_int, out );
}

// ---- BLASInstance::Update on the host (the engine's own restatement; host code, so gcc's contraction is switched off for it)
#define UPD_ATTR __attribute__( (optimize( "fp-contract=off" )) )

/* BLASInstance::InvertTransform (:8402-8428) + Update (:8386-8399).  The frozen reference build vectorises the sixteen cofactor
 * sums, and the lanes of different rows end up with different fused multiply-adds; the shapes below were identified by
 * exhaustive search over every contraction gcc may legally form (3 x 2^4 per cofactor, 12 for the determinant, 6^4 for the
 * corner transform) against BLASInstance::Update on 2,000 random matrices, and are pinned by the tests.  A cofactor is
 * s0*(a0*b0)*c0 + ... + s5*(a5*b5)*c5 with p_k = round( a_k*b_k ):
 *   rows 0,1 : t0 = round( p0*c0 ); acc = fma( +-p1, c1, t0 ); then fma( +-p_k, c_k, acc ) for k = 2..5
 *   row 2    : acc = fma( p0, c0, +-round( p1*c1 ) ); k=2: acc +- round( p2*c2 ); k=3,4: fma; k=5: acc +- round( p5*c5 )
 *   row 3    : acc = fma( p0, c0, +-round( p1*c1 ) ); k=2: fma; k=3,4: acc +- round(..); k=5: fma
 *   det      = fma( T3, c12, fma( T2, c8, fma( T0, c0, round( T1*c4 ) ) ) ); every cell is then multiplied by 1/det
 *   corner   : row = fma( Tz, z, fma( Tx, x, round( Ty*y ) ) ) + Tw, divided by w only when w != 1 */
typedef struct { signed char s; unsigned char a, b, c; } UPD_TERM;
static const UPD_TERM UPD_E[16][6] = {
 {{+1,5,10,15},{-1,5,11,14},{-1,9,6,15},{+1,9,7,14},{+1,13,6,11},{-1,13,7,10}}, {{-1,1,10,15},{+1,1,11,14},{+1,9,2,15},{-1,9,3,14},{-1,13,2,11},{+1,13,3,10}},
 {{+1,1,6,15},{-1,1,7,14},{-1,5,2,15},{+1,5,3,14},{+1,13,2,7},{-1,13,3,6}}, {{-1,1,6,11},{+1,1,7,10},{+1,5,2,11},{-1,5,3,10},{-1,9,2,7},{+1,9,3,6}},
 {{-1,4,10,15},{+1,4,11,14},{+1,8,6,15},{-1,8,7,14},{-1,12,6,11},{+1,12,7,10}}, {{+1,0,10,15},{-1,0,11,14},{-1,8,2,15},{+1,8,3,14},{+1,12,2,11},{-1,12,3,10}},
 {{-1,0,6,15},{+1,0,7,14},{+1,4,2,15},{-1,4,3,14},{-1,12,2,7},{+1,12,3,6}}, {{+1,0,6,11},{-1,0,7,10},{-1,4,2,11},{+1,4,3,10},{+1,8,2,7},{-1,8,3,6}},
 {{+1,4,9,15},{-1,4,11,13},{-1,8,5,15},{+1,8,7,13},{+1,12,5,11},{-1,12,7,9}}, {{-1,0,9,15},{+1,0,11,13},{+1,8,1,15},{-1,8,3,13},{-1,12,1,11},{+1,12,3,9}},
 {{+1,0,5,15},{-1,0,7,13},{-1,4,1,15},{+1,4,3,13},{+1,12,1,7},{-1,12,3,5}}, {{-1,0,5,11},{+1,0,7,9},{+1,4,1,11},{-1,4,3,9},{-1,8,1,7},{+1,8,3,5}},
 {{-1,4,9,14},{+1,4,10,13},{+1,8,5,14},{-1,8,6,13},{-1,12,5,10},{+1,12,6,9}}, {{+1,0,9,14},{-1,0,10,13},{-1,8,1,14},{+1,8,2,13},{+1,12,1,10},{-1,12,2,9}},
 {{-1,0,5,14},{+1,0,6,13},{+1,4,1,14},{-1,4,2,13},{-1,12,1,6},{+1,12,2,5}}, {{+1,0,5,10},{-1,0,6,9},{-1,4,1,10},{+1,4,2,9},{+1,8,1,6},{-1,8,2,5}} };
UPD_ATTR static float upd_cofactor( const float* T, const UPD_TERM* e, const int first_fused_left, const unsigned fused_mask )
{
	float p[6];
	for (int k = 0; k < 6; k++) p[k] = T[e[k].a] * T[e[k].b];
	const float p0 = e[0].s < 0 ? -p[0] : p[0];
	float acc;
	if (first_fused_left) { const float t1 = p[1] * T[e[1].c]; acc = fmaf( p0, T[e[0].c], e[1].s > 0 ? t1 : -t1 ); }
	else { const float t0 = p0 * T[e[0].c]; acc = fmaf( e[1].s > 0 ? p[1] : -p[1], T[e[1].c], t0 ); }
	for (int k = 2; k < 6; k++)
	{
		if (fused_mask & (1u << (k - 2))) acc = fmaf( e[k].s > 0 ? p[k] : -p[k], T[e[k].c], acc );
		else { const float t = p[k] * T[e[k].c]; acc = e[k].s > 0 ? acc + t : acc - t; }
	}
	return acc;
}
UPD_ATTR static void upd_instance( float* T /* transform, 16 */, float* iT /* invTransform, 16 */, float* aabbMin, float* aabbMax, const float* bmin, const float* bmax )
{
	float c[16];
	for (int k = 0; k < 16; k++) c[k] = k < 8 ? upd_cofactor( T, UPD_E[k], 0, 15u ) : k < 12 ? upd_cofactor( T, UPD_E[k], 1, 6u ) : upd_cofactor( T, UPD_E[k], 1, 9u );
	const float t14 = T[1] * c[4];
	const float det = fmaf( T[3], c[12], fmaf( T[2], c[8], fmaf( T[0], c[0], t14 ) ) );
	if (det == 0) { for (int k = 0; k < 16; k++) iT[k] = c[k]; } /* "invert failed": the reference returns with the cofactors stored */
	else { const float invdet = 1.0f / det; for (int k = 0; k < 16; k++) iT[k] = c[k] * invdet; }
	for (int k = 0; k < 3; k++) aabbMin[k] = 1e30f, aabbMax[k] = -1e30f;
	for (int j = 0; j < 8; j++)
	{
		const float p[3] = { j & 1 ? bmax[0] : bmin[0], j & 2 ? bmax[1] : bmin[1], j & 4 ? bmax[2] : bmin[2] };
		float r[3];
		for (int k = 0; k < 3; k++) { const float ty = T[k * 4 + 1] * p[1]; r[k] = fmaf( T[k * 4 + 2], p[2], fmaf( T[k * 4], p[0], ty ) ) + T[k * 4 + 3]; }
		const float wy = T[13] * p[1];
		const float w = fmaf( T[14], p[2], fmaf( T[12], p[0], wy ) ) + T[15];
		if (!(w == 1)) { const float rw = 1.0f / w; r[0] = r[0] * rw, r[1] = r[1] * rw, r[2] = r[2] * rw; }
		for (int k = 0; k < 3; k++) aabbMin[k] = aabbMin[k] < r[k] ? aabbMin[k] : r[k], aabbMax[k] = aabbMax[k] > r[k] ? aabbMax[k] : r[k];
	}
}
#undef UPD_ATTR
int tbvh_instance_update_box( void* instance, const float* bmin, const float* bmax )
{
	ARG_CHECK( instance && bmin && bmax, "NULL argument" );
	float T[16], iT[16], mn[3], mx[3];
	memcpy( T, instance, 64 );
	upd_instance( T, iT, mn, mx, bmin, bmax );
	memcpy( (char*)instance + 64, iT, 64 ), memcpy( (char*)instance + 128, mn, 12 ), memcpy( (char*)instance + 144, mx, 12 );
	return TBVH_OK;
}
int tbvh_instance_update( void* instance, tbvh_bvh blas )
{
	ARG_CHECK( instance && blas, "NULL argument" );
	if (!(blas->info.layouts & (1u << TBVH_LAYOUT_BVH))) { tbvh_set_error( "tbvh_instance_update: the BLAS holds no tree" ); return TBVH_E_STATE; }
	return tbvh_instance_update_box( instance, blas->info.aabb_min, blas->info.aabb_max );
}

// BVH::Build( BLASInstance*, instCount, BVHBase**, blasCount ) tiny_bvh.h:2221 in its "blasses == 0" mode (:2245): the instances
// arrive Update()d - inverse transform and world-space box filled in - and the TLAS is the reference builder's tree over the boxes
int tbvh_build_tlas( tbvh_bvh t, const void* instances, uint32_t inst_stride, uint32_t inst_count, const tbvh_bvh* blasses, uint32_t blas_count, float c_trav, float c_int )
{
	ARG_CHECK( t && instances && blasses && inst_count > 0 && blas_count > 0 && inst_stride >= 160, "bad TLAS arguments" );
	CUDA_TRY( cudaSetDevice( t->ctx->device ) );
	free_layouts( t );
	std::vector<float4> boxes( (size_t)inst_count * 2 );
	std::vector<TlasInst> inst( inst_count );
	std::vector<BlasRef> refs( blas_count );
	uint32_t blas_layouts = (1u << TBVH_LAYOUT_BVH) | (1u << TBVH_LAYOUT_CWBVH);
	for (uint32_t k = 0; k < blas_count; k++)
	{
		const tbvh_bvh b = blasses[k];
		ARG_CHECK( b && b != t && b->ctx == t->ctx, "TLAS: a BLAS handle is NULL or lives in another context" );
		const bool has_bvh = (b->info.layouts & (1u << TBVH_LAYOUT_BVH)) && b->d_trav && b->d_leaf_tris, has_cw = b->d_cw_trav && b->d_cw_tris;
		if (b->d_inst || (!has_bvh && !has_cw))
		{ tbvh_set_error( "TLAS: BLAS %u holds no triangle tree (IntersectTLAS walks LAYOUT_BVH BLASses, tiny_bvh.h:3341; traverse_tlas.cl CWBVH ones)", k ); return TBVH_E_STATE; }
		if (has_bvh && b->info.max_depth + 1 > TBVH_STACK) { tbvh_set_error( "TLAS: BLAS %u has depth %u, the two-level kernel walks a BLAS with a %d-entry stack", k, b->info.max_depth, TBVH_STACK ); return TBVH_E_LIMIT; }
		if (has_cw && b->cw_depth + 1 > 128) { tbvh_set_error( "TLAS: the wide tree of BLAS %u has depth %u (128 pending node groups per ray, tiny_bvh.h:7048)", k, b->cw_depth ); return TBVH_E_LIMIT; }
		refs[k].trav = has_bvh ? b->d_trav : 0, refs[k].tris = has_bvh ? b->d_leaf_tris : 0, refs[k].root_ref = b->root_ref, refs[k].root_count = b->root_count, refs[k].pad0 = refs[k].pad1 = 0;
		refs[k].cw_nodes = has_cw ? b->d_cw_trav : 0, refs[k].cw_tris = has_cw ? b->d_cw_tris : 0;
		blas_layouts &= (has_bvh ? 1u << TBVH_LAYOUT_BVH : 0u) | (has_cw ? 1u << TBVH_LAYOUT_CWBVH : 0u);
	}
	for (uint32_t i = 0; i < inst_count; i++)
	{
		// BLASInstance :1443: transform @0, invTransform @64, aabbMin @128, blasIdx @140, aabbMax @144, mask @156
		const char* r = (const char*)instances + (size_t)i * inst_stride;
		memcpy( inst[i].inv, r + 64, 64 );
		memcpy( &inst[i].blasIdx, r + 140, 4 ), memcpy( &inst[i].mask, r + 156, 4 );
		inst[i].pad0 = inst[i].pad1 = 0;
		ARG_CHECK( inst[i].blasIdx < blas_count, "TLAS: an instance names a BLAS past blas_count" );
		float mn[3], mx[3];
		memcpy( mn, r + 128, 12 ), memcpy( mx, r + 144, 12 );
		boxes[(size_t)i * 2] = make_float4( mn[0], mn[1], mn[2], 0 ), boxes[(size_t)i * 2 + 1] = make_float4( mx[0], mx[1], mx[2], 0 );
	}
	cudaStream_t s = t->ctx->stream;
	CUDA_TRY( cudaMalloc( &t->d_aabbs, boxes.size() * 16 ) );
	CUDA_TRY( cudaMalloc( &t->d_inst, inst.size() * sizeof( TlasInst ) ) );
	CUDA_TRY( cudaMalloc( &t->d_blas, refs.size() * sizeof( BlasRef ) ) );
	CUDA_TRY( cudaMemcpyAsync( t->d_aabbs, boxes.data(), boxes.size() * 16, cudaMemcpyHostToDevice, s ) );
	CUDA_TRY( cudaMemcpyAsync( t->d_inst, inst.data(), inst.size() * sizeof( TlasInst ), cudaMemcpyHostToDevice, s ) );
	CUDA_TRY( cudaMemcpyAsync( t->d_blas, refs.data(), refs.size() * sizeof( BlasRef ), cudaMemcpyHostToDevice, s ) );
	CUDA_TRY( cudaStreamSynchronize( s ) ); // the host vectors go out of scope
	t->info.prim_count = inst_count, t->inst_count = inst_count, t->blas_count = blas_count, t->tlas_blas_layouts = blas_layouts;
	TRY( build_sah_launch( t, c_trav, c_int, TBVH_BUILD_REFERENCE ) ); // "Build(); // or BuildAVX, for large TLAS." :2258
	t->info.layouts = 1u << TBVH_LAYOUT_BVH, t->refittable = false; // "do not refit a TLAS, use Build(..)" :3060
	if (t->info.max_depth + 1 > TBVH_STACK) { tbvh_set_error( "TLAS depth %u exceeds the %d-entry stack of IntersectTLAS (tiny_bvh.h:3308)", t->info.max_depth, TBVH_STACK ); return TBVH_E_LIMIT; }
	// the device table holds raw addresses of the BLAS arrays: remember which generation of each BLAS they belong to
	for (uint32_t k = 0; k < blas_count; k++) t->links.push_back( BlasLink{ blasses[k], blasses[k]->generation } );
	return TBVH_OK;
}

// BVH::Refit (tiny_bvh.h:3055): same topology, new vertex positions
int tbvh_refit( tbvh_bvh b, const void* verts, uint32_t stride, uint32_t prim_count, int space )
{
	ARG_CHECK( b && verts, "NULL argument" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	if (!(b->info.layouts & (1u << TBVH_LAYOUT_BVH)) || !b->d_nodes || b->d_trav != b->d_nodes) { tbvh_set_error( "tbvh_refit: no BVH-layout tree on this handle" ); return TBVH_E_STATE; }
	if (!b->refittable) { tbvh_set_error( "tbvh_refit: refitting an SBVH (BVH::Refit, tiny_bvh.h:3057)" ); return TBVH_E_STATE; }
	ARG_CHECK( prim_count == b->info.prim_count && stride >= 12 && (stride & 3) == 0, "tbvh_refit: the vertex slice must describe the same triangles" );
	cudaStream_t s = b->ctx->stream;
	const size_t nv = (size_t)prim_count * 3;
	const cudaMemcpyKind kind = space == TBVH_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	if (stride == 16) CUDA_TRY( cudaMemcpyAsync( b->d_verts, verts, nv * 16, kind, s ) );
	else CUDA_TRY( cudaMemcpy2DAsync( b->d_verts, 16, verts, stride, stride < 16 ? stride : 16, nv, kind, s ) );
	TRY( refit_launch( b, s ) );
	// derived layouts describe the old boxes: drop them (the reference's BVH_GPU / BVH8_CWBVH are re-converted after a refit too)
	if (b->d_nodes_gpu) cudaFree( b->d_nodes_gpu ), b->d_nodes_gpu = 0;
	if (b->d_cw_trav || b->d_cw_tris) b->generation = tbvh_next_generation(); // a TLAS may hold these addresses (tlas_check)
	if (b->d_cw_nodes) cudaFree( b->d_cw_nodes ), b->d_cw_nodes = 0;
	if (b->d_cw_tris) cudaFree( b->d_cw_tris ), b->d_cw_tris = 0;
	if (b->d_cw_trav) cudaFree( b->d_cw_trav ), b->d_cw_trav = 0;
	b->info.layouts = 1u << TBVH_LAYOUT_BVH, b->info.used_nodes_gpu = 0, b->info.used_blocks = 0, b->info.cwbvh_tri_count = 0;
	TRY( make_leaf_tris( b, s ) );
	CUDA_TRY( cudaStreamSynchronize( s ) );
	return TBVH_OK;
}

int tbvh_build_indexed( tbvh_bvh b, const void* verts, uint32_t stride, uint32_t vert_count, const uint32_t* indices, uint32_t prim_count, int space,
	float c_trav, float c_int, int flavour )
{
	ARG_CHECK( b, "NULL handle" );
	ARG_CHECK( flavour == TBVH_BUILD_REFERENCE || flavour == TBVH_BUILD_AVX || flavour == TBVH_BUILD_HQ, "unknown builder flavour" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	free_layouts( b );
	TRY( upload_verts_indexed( b, verts, stride, vert_count, indices, prim_count, space, b->ctx->stream ) );
	if (flavour == TBVH_BUILD_HQ) TRY( build_hq_launch( b, c_trav, c_int ) ); else TRY( build_sah_launch( b, c_trav, c_int, flavour ) );
	b->info.layouts = 1u << TBVH_LAYOUT_BVH, b->refittable = flavour != TBVH_BUILD_HQ;
	return TBVH_OK;
}

int tbvh_build( tbvh_bvh b, const void* verts, uint32_t stride, uint32_t prim_count, int space, float c_trav, float c_int )
{
	return tbvh_build_flavour( b, verts, stride, prim_count, space, c_trav, c_int, TBVH_BUILD_REFERENCE );
}

int tbvh_convert( tbvh_bvh b, int to_layout )
{
	ARG_CHECK( b, "NULL handle" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	if (!(b->info.layouts & (1u << TBVH_LAYOUT_BVH))) { tbvh_set_error( "tbvh_convert: source layout BVH not resident" ); return TBVH_E_STATE; }
	if (to_layout == TBVH_LAYOUT_BVH_GPU) { TRY( bvh_to_bvh_gpu( b, b->ctx->stream ) ); b->info.layouts |= 1u << TBVH_LAYOUT_BVH_GPU; return TBVH_OK; }
	if (to_layout == TBVH_LAYOUT_CWBVH) { TRY( bvh_to_cwbvh( b, b->ctx->stream ) ); b->info.layouts |= 1u << TBVH_LAYOUT_CWBVH; return TBVH_OK; }
	tbvh_set_error( "tbvh_convert: unsupported target layout %d", to_layout );
	return TBVH_E_UNSUPPORTED;
}

static cudaMemcpyKind out_kind( int space ) { return space == TBVH_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost; }

int tbvh_download_bvh( tbvh_bvh b, void* nodes32, uint32_t* prim_idx, int space )
{
	ARG_CHECK( b, "NULL handle" );
	if (!(b->info.layouts & (1u << TBVH_LAYOUT_BVH))) { tbvh_set_error( "layout BVH not resident" ); return TBVH_E_STATE; }
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	if (nodes32) CUDA_TRY( cudaMemcpy( nodes32, b->d_nodes, (size_t)b->info.used_nodes * 32, out_kind( space ) ) );
	if (prim_idx) CUDA_TRY( cudaMemcpy( prim_idx, b->d_prim_idx, (size_t)b->info.idx_count * 4, out_kind( space ) ) );
	return TBVH_OK;
}

int tbvh_download_bvh_gpu( tbvh_bvh b, void* nodes64, int space )
{
	ARG_CHECK( b && nodes64, "NULL argument" );
	if (!(b->info.layouts & (1u << TBVH_LAYOUT_BVH_GPU)) || !b->d_nodes_gpu) { tbvh_set_error( "layout BVH_GPU not resident" ); return TBVH_E_STATE; }
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	CUDA_TRY( cudaMemcpy( nodes64, b->d_nodes_gpu, (size_t)b->info.used_nodes_gpu * 64, out_kind( space ) ) );
	return TBVH_OK;
}

int tbvh_download_cwbvh( tbvh_bvh b, void* bvh8_data, void* bvh8_tris, int space )
{
	ARG_CHECK( b, "NULL handle" );
	if (!(b->info.layouts & (1u << TBVH_LAYOUT_CWBVH))) { tbvh_set_error( "layout CWBVH not resident" ); return TBVH_E_STATE; }
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	if (bvh8_data) CUDA_TRY( cudaMemcpy( bvh8_data, b->d_cw_nodes, (size_t)b->info.used_blocks * 16, out_kind( space ) ) );
	if (bvh8_tris) CUDA_TRY( cudaMemcpy( bvh8_tris, b->d_cw_tris, (size_t)b->info.cwbvh_tri_count * 48, out_kind( space ) ) );
	return TBVH_OK;
}

// ---- traversal ------------------------------------------------------------------------------------------------

// live handles (a TLAS remembers its BLAS handles; a destroyed one must be noticed, not dereferenced)
static std::mutex g_live_mutex;
static std::vector<tbvh_bvh> g_live;
static void live_add( tbvh_bvh b ) { std::lock_guard<std::mutex> lk( g_live_mutex ); g_live.push_back( b ); }
static void live_remove( tbvh_bvh b ) { std::lock_guard<std::mutex> lk( g_live_mutex ); for (size_t i = 0; i < g_live.size(); i++) if (g_live[i] == b) { g_live[i] = g_live.back(); g_live.pop_back(); break; } }

// a TLAS points at the arrays of its BLASses: refuse to walk it once one of them was rebuilt, re-uploaded or destroyed
static int tlas_check( tbvh_bvh t, int layout )
{
	// the layout argument of a traversal call on a TLAS names the layout the BLASses are walked in (trace_tlas.cu)
	const uint32_t want = layout == TBVH_LAYOUT_CWBVH ? 1u << TBVH_LAYOUT_CWBVH : 1u << TBVH_LAYOUT_BVH;
	if (layout != TBVH_LAYOUT_CWBVH && layout != TBVH_LAYOUT_BVH && layout != TBVH_LAYOUT_BVH_GPU) { tbvh_set_error( "unknown layout %d", layout ); return TBVH_E_ARG; }
	if (!(t->tlas_blas_layouts & want))
	{ tbvh_set_error( "TLAS: not every BLAS held its %s layout when the TLAS was built", layout == TBVH_LAYOUT_CWBVH ? "CWBVH" : "BVH" ); return TBVH_E_STATE; }
	std::lock_guard<std::mutex> lk( g_live_mutex );
	for (const BlasLink& l : t->links)
	{
		bool alive = false;
		for (tbvh_bvh h : g_live) if (h == l.blas) { alive = true; break; }
		if (!alive || l.blas->generation != l.generation)
		{ tbvh_set_error( "TLAS is stale: a BLAS it was built over has been %s since (build the TLAS again, tiny_bvh.h:2221)", alive ? "rebuilt or re-uploaded" : "destroyed" ); return TBVH_E_STATE; }
	}
	return TBVH_OK;
}

static int trace_dispatch( tbvh_bvh b, int layout, const void* d_rays, uint32_t stride, void* d_hits, uint32_t hit_stride,
	uint32_t* d_bits, uint64_t n, bool anyhit, cudaStream_t s )
{
	unsigned long long* st = b->stats ? b->d_stats : 0;
	if (layout == TBVH_LAYOUT_BVH || layout == TBVH_LAYOUT_BVH_GPU) return bvh2_trace_launch( b, d_rays, stride, d_hits, hit_stride, d_bits, n, anyhit, s, st );
	if (layout == TBVH_LAYOUT_CWBVH) return cwbvh_trace_launch( b, d_rays, stride, d_hits, hit_stride, d_bits, n, anyhit, s, st );
	tbvh_set_error( "unknown layout %d", layout );
	return TBVH_E_ARG;
}

int tbvh_intersect_device( tbvh_bvh b, int layout, void* d_rays, uint32_t stride, void* d_hits, uint64_t n, void* stream )
{
	ARG_CHECK( b && d_rays && stride >= 64 && (stride & 15) == 0, "bad ray buffer" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	if (b->stats) CUDA_TRY( cudaMemsetAsync( b->d_stats, 0, 32, (cudaStream_t)stream ) );
	if (b->d_inst)
	{
		// TLAS: hits carry the instance (hit.inst, byte 44) and are written into the ray records
		if (d_hits) { tbvh_set_error( "TLAS hits are written in place (t,u,v,prim at byte 48, inst at byte 44): pass d_hits = NULL" ); return TBVH_E_UNSUPPORTED; }
		TRY( tlas_check( b, layout ) );
		return tlas_trace_launch( b, layout, d_rays, stride, 0, n, false, (cudaStream_t)stream );
	}
	if (d_hits) return trace_dispatch( b, layout, d_rays, stride, d_hits, 16, 0, n, false, (cudaStream_t)stream );
	return trace_dispatch( b, layout, d_rays, stride, (char*)d_rays + 48, stride, 0, n, false, (cudaStream_t)stream );
}

int tbvh_occluded_device( tbvh_bvh b, int layout, const void* d_rays, uint32_t stride, uint32_t* d_bits, uint64_t n, void* stream )
{
	ARG_CHECK( b && d_rays && d_bits && stride >= 64 && (stride & 15) == 0, "bad ray buffer" );
	CUDA_TRY( cudaSetDevice( b->ctx->device ) );
	if (b->stats) CUDA_TRY( cudaMemsetAsync( b->d_stats, 0, 32, (cudaStream_t)stream ) );
	if (b->d_inst) { TRY( tlas_check( b, layout ) ); return tlas_trace_launch( b, layout, d_rays, stride, d_bits, n, true, (cudaStream_t)stream ); }
	return trace_dispatch( b, layout, d_rays, stride, 0, 0, d_bits, n, true, (cudaStream_t)stream );
}

// plain device memory for callers of the *_device entry points that do not link the CUDA runtime themselves
int tbvh_device_alloc( tbvh_ctx c, size_t bytes, void** out )
{
	ARG_CHECK( c && out, "NULL argument" );
	CUDA_TRY( cudaSetDevice( c->device ) );
	CUDA_TRY( cudaMalloc( out, bytes ) );
	return TBVH_OK;
}
int tbvh_device_free( tbvh_ctx c, void* p )
{
	ARG_CHECK( c, "NULL context" );
	CUDA_TRY( cudaSetDevice( c->device ) );
	if (p) CUDA_TRY( cudaFree( p ) );
	return TBVH_OK;
}
int tbvh_device_sync( tbvh_ctx c )
{
	ARG_CHECK( c, "NULL context" );
	CUDA_TRY( cudaSetDevice( c->device ) );
	CUDA_TRY( cudaDeviceSynchronize() );
	return TBVH_OK;
}
int tbvh_copy_from_device( void* host, const void* d_src, size_t bytes )
{
	ARG_CHECK( host && d_src, "NULL argument" );
	CUDA_TRY( cudaMemcpy( host, d_src, bytes, cudaMemcpyDeviceToHost ) );
	return TBVH_OK;
}

// host records -> packed 64-byte device records (bytes 0..63 of each), asynchronous on `stream`: what a caller of the *_device
// entry points needs to get its batch into HBM (the speedtest's own upload, tiny_bvh_speedtest.cpp:1110-1115)
int tbvh_copy_rays_to_device( const void* rays, uint32_t stride, uint64_t n, void* d_rays, void* stream )
{
	ARG_CHECK( rays && d_rays && stride >= 64, "bad ray buffer" );
	if (n == 0) return TBVH_OK;
	CUDA_TRY( cudaMemcpy2DAsync( d_rays, 64, rays, stride, 64, n, cudaMemcpyHostToDevice, (cudaStream_t)stream ) );
	return TBVH_OK;
}

// ---- host-buffer path ---------------------------------------------------------------------------------------------
// tbvh_intersect / tbvh_intersect_packed / tbvh_occluded on HOST ray records.  Only bytes 0..63 of each record cross PCIe inbound,
// and outbound only what the call returns.  The batch is cut into chunks that flow through TBVH_SLOTS stage buffers:
//
//     s_in  : chunk k+1   host records --(2D copy of 64-byte rows)--> slot.d_rays
//     s_run : chunk k     traversal kernel: hits into the staged records (in place, TLAS) or slot.d_hits (packed) / slot.d_bits
//     s_out : chunk k-1   back to the host: bytes 0..63 of every record (in place), one contiguous copy (packed), 20-byte rows at
//                         byte 44 (TLAS: instance + hit) or the occlusion words
//
// Each direction owns a stream, so the inbound copy engine never waits for an outbound copy queued ahead of it; events hand a
// slot from stage to stage and back (out_done -> the next inbound copy into that slot).  One call at a time per context
// (host_mutex): concurrent callers on one handle are serialised, as SURVEY 8(b) asks.
static int ensure_slots( tbvh_ctx c )
{
	// allocated once; a call that failed half-way leaves the buffers it got, and the next one completes the set
	for (HostSlot& sl : c->slot)
	{
		if (!sl.d_rays) CUDA_TRY( cudaMalloc( &sl.d_rays, (size_t)TBVH_CHUNK_RAYS * 64 ) );
		if (!sl.d_hits) CUDA_TRY( cudaMalloc( &sl.d_hits, (size_t)TBVH_CHUNK_RAYS * 16 ) );
		if (!sl.d_bits) CUDA_TRY( cudaMalloc( &sl.d_bits, TBVH_CHUNK_RAYS / 8 + 4 ) );
	}
	return TBVH_OK;
}

// inbound stage of one chunk: on return s_in carries the copy and slot.in_done is recorded behind it
static int stage_in( tbvh_ctx c, const uint64_t chunk, const char* h, const uint32_t stride, const uint64_t cnt )
{
	HostSlot& sl = c->slot[chunk % TBVH_SLOTS];
	if (chunk >= TBVH_SLOTS) CUDA_TRY( cudaStreamWaitEvent( c->s_in, sl.out_done, 0 ) ); // the slot's previous tenant has left the device
	CUDA_TRY( cudaMemcpy2DAsync( sl.d_rays, 64, h, stride, 64, cnt, cudaMemcpyHostToDevice, c->s_in ) );
	CUDA_TRY( cudaEventRecord( sl.in_done, c->s_in ) );
	CUDA_TRY( cudaStreamWaitEvent( c->s_run, sl.in_done, 0 ) );
	return TBVH_OK;
}

static int drain( tbvh_ctx c )
{
	CUDA_TRY( cudaStreamSynchronize( c->s_out ) );
	CUDA_TRY( cudaStreamSynchronize( c->s_run ) );
	CUDA_TRY( cudaStreamSynchronize( c->s_in ) );
	return TBVH_OK;
}

static int intersect_host( tbvh_bvh b, int layout, void* rays, uint32_t stride, uint64_t n, void* packed_hits )
{
	ARG_CHECK( b && rays && stride >= 64, "bad ray buffer" );
	tbvh_ctx c = b->ctx;
	std::lock_guard<std::mutex> lk( c->host_mutex );
	CUDA_TRY( cudaSetDevice( c->device ) );
	TRY( ensure_slots( c ) );
	if (b->stats) CUDA_TRY( cudaMemset( b->d_stats, 0, 32 ) );
	const bool tlas = b->d_inst != 0;
	if (tlas)
	{
		if (packed_hits) { tbvh_set_error( "tbvh_intersect_packed: TLAS hits carry the instance and are returned in the ray records" ); return TBVH_E_UNSUPPORTED; }
		TRY( tlas_check( b, layout ) );
	}
	uint64_t chunk = 0;
	int rc = TBVH_OK;
	for (uint64_t off = 0; off < n && rc == TBVH_OK; off += TBVH_CHUNK_RAYS, chunk++)
	{
		HostSlot& sl = c->slot[chunk % TBVH_SLOTS];
		const uint64_t cnt = n - off < TBVH_CHUNK_RAYS ? n - off : TBVH_CHUNK_RAYS;
		char* h = (char*)rays + off * stride;
		auto body = [&]() -> int
		{
			TRY( stage_in( c, chunk, h, stride, cnt ) );
			// in place, the kernel writes the hit into the staged record and bytes 0..63 of every record - exactly its first cache line -
			// travel back, so the host receives FULL-line writes (no read-for-ownership of a partially written line); bytes 0..47 return
			// unchanged.  A TLAS writes hit + instance into the staged records as well.
			if (tlas) TRY( tlas_trace_launch( b, layout, sl.d_rays, 64, 0, cnt, false, c->s_run ) );
			else if (packed_hits) TRY( trace_dispatch( b, layout, sl.d_rays, 64, sl.d_hits, 16, 0, cnt, false, c->s_run ) );
			else TRY( trace_dispatch( b, layout, sl.d_rays, 64, (char*)sl.d_rays + 48, 64, 0, cnt, false, c->s_run ) );
			CUDA_TRY( cudaEventRecord( sl.run_done, c->s_run ) );
			CUDA_TRY( cudaStreamWaitEvent( c->s_out, sl.run_done, 0 ) );
			if (tlas) CUDA_TRY( cudaMemcpy2DAsync( h + 44, stride, (char*)sl.d_rays + 44, 64, 20, cnt, cudaMemcpyDeviceToHost, c->s_out ) );
			else if (packed_hits) CUDA_TRY( cudaMemcpyAsync( (char*)packed_hits + off * 16, sl.d_hits, cnt * 16, cudaMemcpyDeviceToHost, c->s_out ) );
			else CUDA_TRY( cudaMemcpy2DAsync( h, stride, sl.d_rays, 64, 64, cnt, cudaMemcpyDeviceToHost, c->s_out ) );
			CUDA_TRY( cudaEventRecord( sl.out_done, c->s_out ) );
			return TBVH_OK;
		};
		rc = body();
	}
	const int rd = drain( c ); // also after an error: nothing of this call may still be in flight when the mutex is released
	return rc != TBVH_OK ? rc : rd;
}

int tbvh_intersect( tbvh_bvh b, int layout, void* rays, uint32_t stride, uint64_t n ) { return intersect_host( b, layout, rays, stride, n, 0 ); }

int tbvh_intersect_packed( tbvh_bvh b, int layout, const void* rays, uint32_t stride, uint64_t n, void* hits )
{
	ARG_CHECK( hits, "hits == NULL" );
	return intersect_host( b, layout, (void*)rays, stride, n, hits );
}

int tbvh_occluded( tbvh_bvh b, int layout, const void* rays, uint32_t stride, uint64_t n, uint32_t* bits )
{
	ARG_CHECK( b && rays && bits && stride >= 64, "bad ray buffer" );
	tbvh_ctx c = b->ctx;
	std::lock_guard<std::mutex> lk( c->host_mutex );
	CUDA_TRY( cudaSetDevice( c->device ) );
	TRY( ensure_slots( c ) );
	if (b->stats) CUDA_TRY( cudaMemset( b->d_stats, 0, 32 ) );
	if (b->d_inst) TRY( tlas_check( b, layout ) );
	uint64_t chunk = 0;
	int rc = TBVH_OK;
	for (uint64_t off = 0; off < n && rc == TBVH_OK; off += TBVH_CHUNK_RAYS, chunk++)
	{
		HostSlot& sl = c->slot[chunk % TBVH_SLOTS];
		const uint64_t cnt = n - off < TBVH_CHUNK_RAYS ? n - off : TBVH_CHUNK_RAYS;
		const char* h = (const char*)rays + off * stride;
		auto body = [&]() -> int
		{
			TRY( stage_in( c, chunk, h, stride, cnt ) );
			if (b->d_inst) TRY( tlas_trace_launch( b, layout, sl.d_rays, 64, (uint32_t*)sl.d_bits, cnt, true, c->s_run ) );
			else TRY( trace_dispatch( b, layout, sl.d_rays, 64, 0, 0, (uint32_t*)sl.d_bits, cnt, true, c->s_run ) );
			CUDA_TRY( cudaEventRecord( sl.run_done, c->s_run ) );
			CUDA_TRY( cudaStreamWaitEvent( c->s_out, sl.run_done, 0 ) );
			CUDA_TRY( cudaMemcpyAsync( bits + off / 32, sl.d_bits, ((cnt + 31) / 32) * 4, cudaMemcpyDeviceToHost, c->s_out ) ); // TBVH_CHUNK_RAYS is a multiple of 32
			CUDA_TRY( cudaEventRecord( sl.out_done, c->s_out ) );
			return TBVH_OK;
		};
		rc = body();
	}
	const int rd = drain( c );
	return rc != TBVH_OK ? rc : rd;
}

} // extern "C"
