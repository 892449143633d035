// ufo_map.cu -- host side of libufomap_b200.so: device pools, scan orchestration
// and the C ABI declared in include/ufomap_b200.h.
//
// One map = one CUDA device + one stream (+ a copy stream for the points).  An insert enqueues
//   H2D(points) -> K1 k_points [-> K1b k_hits] -> k_split -> k_walk_mark -> k_gather_scan ->
//   k_gather -> K3 k_update_brick -> K4 k_upper_* -> D2H(counters)
// and returns; the next call that looks at the map reads the counters, grows a pool and repeats
// the scan if an allocation overflowed (finalize_scan).  Insert depth >= 3, maps that have seen
// out-of-tree keys and the fixed-step walk use k_rays -> k_scatter instead of the fused walk,
// which mirrors insertPointCloud + insertPointCloudHelper
// (/root/reference/ufomap/include/ufo/map/occupancy_map_base.h:270-327, :1345-1373).
// There is no CPU fallback anywhere in this file.

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <numeric>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/ufomap_b200.h"
#include "ufo_kernels.cuh"
#include "ufo_export.cuh"
#include "ufo_walk.cuh"
#include "ufo_route.cuh"
#include "ufo_import.cuh"

using namespace ufo_b200;

namespace
{
constexpr uint32_t kMinHash = 1u << 16;

uint32_t next_pow2(uint64_t v)
{
	uint64_t p = 1;
	while (p < v) p <<= 1;
	return (uint32_t)std::min<uint64_t>(p, 1ull << 31);
}

struct CudaError {
	cudaError_t e;
	const char* what;
	int line;
};

#define CK(call)                                         \
	do {                                                   \
		cudaError_t e__ = (call);                            \
		if (e__ != cudaSuccess) throw CudaError{e__, #call, __LINE__}; \
	} while (0)

enum class Mem { kDevice, kPinned };

// Owns one allocation of T: device memory, or pinned host memory.  A buffer made with a byte
// count adds its size to it while it holds memory, so that the count is always the sum over the
// owner's live buffers (ufo_b200_scan_stats::device_bytes).
template <class T, Mem kMem = Mem::kDevice>
class Buffer
{
public:
	Buffer(size_t* total = nullptr) : total_(total) {}
	Buffer(Buffer&& o) noexcept : p_(o.p_), n_(o.n_), total_(o.total_)
	{
		o.p_ = nullptr;
		o.n_ = 0;
	}
	Buffer& operator=(Buffer&& o) noexcept
	{
		std::swap(p_, o.p_);
		std::swap(n_, o.n_);
		std::swap(total_, o.total_);
		return *this;
	}
	~Buffer() { reset(); }

	T* get() const { return p_; }
	T* operator->() const { return p_; }
	T& operator*() const { return *p_; }
	size_t size() const { return n_; }
	size_t bytes() const { return n_ * sizeof(T); }

	void reset()
	{
		if (!p_) return;
		if (kMem == Mem::kPinned) cudaFreeHost(p_);
		else cudaFree(p_);
		if (total_) *total_ -= bytes();
		p_ = nullptr;
		n_ = 0;
	}

	// n elements (at least one); the contents are not kept.  fill >= 0: every byte is set to it on s.
	void resize(size_t n, int fill = -1, cudaStream_t s = nullptr)
	{
		reset();
		n = std::max<size_t>(n, 1);
		if (kMem == Mem::kPinned) CK(cudaHostAlloc(reinterpret_cast<void**>(&p_), n * sizeof(T), cudaHostAllocDefault));
		else CK(cudaMalloc(reinterpret_cast<void**>(&p_), n * sizeof(T)));
		n_ = n;
		if (total_) *total_ += bytes();
		if (fill >= 0) CK(cudaMemsetAsync(p_, fill, bytes(), s));
	}

	// n elements, the contents kept and the new part set to fill; waits for s
	void grow(size_t n, int fill, cudaStream_t s)
	{
		Buffer q(total_);
		q.resize(n);
		CK(cudaMemcpyAsync(q.p_, p_, bytes(), cudaMemcpyDeviceToDevice, s));
		CK(cudaMemsetAsync(q.p_ + n_, fill, q.bytes() - bytes(), s));
		CK(cudaStreamSynchronize(s));
		*this = std::move(q);
	}

	// sets the first n elements (all of them by default) to `byte` on s
	void fill(int byte, cudaStream_t s, size_t n = ~size_t(0)) const
	{
		CK(cudaMemsetAsync(p_, byte, std::min(n, n_) * sizeof(T), s));
	}

private:
	T* p_ = nullptr;
	size_t n_ = 0;
	size_t* total_;
};

double to_logit(double p) { return std::log(p / (1.0 - p)); }
}  // namespace

struct MapError {
	int code;
};

// everything needed to enqueue a scan again after a pool growth
struct PendingScan {
	bool valid = false;
	ScanArgs a{};
	bool use_color = false, need_table = false, simple = false, has_vol = false;
	bool routed = false;  // routed multi-GPU pass: cannot be repeated locally after a pool overflow
	bool dense = false;   // marks go to the dense scan volume
	VolumeArgs vol{};
	float set_value = 0.0f;
	uint32_t regrows = 0;
};

struct ufo_b200_map {
	ufo_b200_params params{};
	DeviceMap M{};
	int device = 0;
	cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
	cudaEvent_t ev_copy0 = nullptr, ev_copied = nullptr;
	// sensor model as the reference stores it (double log-odds)
	double occ_thr_log = 0, free_thr_log = 0, hit_log = 0, miss_log = 0, cmin_log = 0, cmax_log = 0;
	// Every allocation of the map is one of the buffers below; device_bytes is the sum of the sizes
	// of the device buffers (each adds and removes its own).
	size_t device_bytes = 0;
	// brick and upper-node pools: one buffer per array of for_each_pool_array, which also points
	// the DeviceMap fields (and the views below) at them
	std::vector<Buffer<unsigned char>> pool;
	uint32_t* d_list[2] = {nullptr, nullptr};  // dirty lists of the upper-level pass
	unsigned long long* chg_mask = nullptr;    // change mask (DeviceMap::chg_mask while recording)
	bool chg_recording = false;
	Buffer<ulonglong2> bh_tab{&device_bytes};
	Buffer<unsigned long long> uh_keys{&device_bytes};
	Buffer<uint32_t> uh_vals{&device_bytes};
	Buffer<Counters> ctr{&device_bytes};
	Buffer<Counters, Mem::kPinned> h_ctr;  // host mirror of the counters
	// scan staging: two point buffers, so that the H2D copy of scan k+1 overlaps scan k
	Buffer<unsigned char> d_points[2] = {&device_bytes, &device_bytes};
	uint32_t stage = 0;
	Buffer<double> d_ray_end{&device_bytes};  // [ray capacity][3]
	Buffer<uint32_t> d_hit_tab{&device_bytes};  // [ray capacity]
	Buffer<unsigned long long> d_tab_keys{&device_bytes};
	Buffer<uint32_t> d_tab_min{&device_bytes};
	// generic marking path: ray-walk records
	Buffer<QEntry> d_seg{&device_bytes};
	Buffer<uint32_t> d_seg_base{&device_bytes}, d_seg_count{&device_bytes}, d_order{&device_bytes};
	Buffer<unsigned long long> d_nodes{&device_bytes};  // insert depth 5/6: free-space nodes of the scan
	// fused walk: segments, validity masks, per-ray constants
	Buffer<Item> d_items{&device_bytes};
	Buffer<uint32_t> d_vmask{&device_bytes};
	Buffer<RayConst> d_rc{&device_bytes};
	// dense scan volume
	Buffer<unsigned long long> vol{&device_bytes}, vol_dirty{&device_bytes};
	Buffer<uint32_t> vol_list{&device_bytes};
	// bookkeeping
	uint32_t n_blocks = 0, n_bricks = 0, n_upper = 0;  // host view after the last completed scan
	int profiling = 0;
	int force_records = 0;  // UFO_B200_MARK=records: always use the record path (A/B runs)
	int k3_blocks = 0;      // UFO_B200_K3_BLOCKS: resident K3 CTAs per SM (0: the kernel's launch bound)
	int no_dense = 0;       // UFO_B200_MARK=probe, or a scan left the volume: fused walk through the brick hash
	uint32_t vol_db_cap = 0;  // bricks per axis the allocated scan volume can hold
	uint64_t launches = 0;
	cudaEvent_t ev[8]{};
	bool ev_valid = false, ev7_valid = false, h2d_valid = false;
	ufo_b200_scan_stats stats{};       // scan in flight / last scan
	ufo_b200_scan_stats done_stats{};  // last scan whose counters are folded into the host view
	bool stats_pending = false;
	PendingScan pending;
	bool poisoned = false;
	// routed multi-GPU mode
	Buffer<unsigned char> route_inbox{&device_bytes};  // this rank's inbox: [2 parities][world sources] regions
	Buffer<RouteTable> route{&device_bytes};
	size_t route_region = 0, route_miss_off = 0, route_hit_off = 0;
	void* route_peer[kMaxRanks] = {};
	Buffer<RouteTable, Mem::kPinned> h_route;  // pinned mirror, pushed before every mark pass
	Buffer<uint32_t, Mem::kPinned> h_route_flag;
	uint32_t route_parity = 0, route_cap_m = 0, route_cap_h = 0;
	int route_stage = 0;  // 0 idle, 1 marked (waiting for the apply calls), 2 applied
	double min_change[3], max_change[3];
	std::string err;
	int sm_count = 148;
	int ray_blocks_per_sm = 4, walk_blocks_per_sm = 4;

	// the buffers free themselves after this; the caller has waited for the stream
	~ufo_b200_map()
	{
		for (cudaEvent_t e : ev)
			if (e) cudaEventDestroy(e);
		if (ev_copy0) cudaEventDestroy(ev_copy0);
		if (ev_copied) cudaEventDestroy(ev_copied);
		if (own_stream) cudaStreamDestroy(own_stream);
		if (copy_stream) cudaStreamDestroy(copy_stream);
	}

	void set_error(const char* fmt, ...)
	{
		char buf[512];
		va_list ap;
		va_start(ap, fmt);
		vsnprintf(buf, sizeof(buf), fmt, ap);
		va_end(ap);
		err = buf;
	}
};

namespace
{
using Map = ufo_b200_map;

void refresh_model(Map* m)
{
	DeviceMap& M = m->M;
	M.occ_thr = m->occ_thr_log;
	M.free_thr = m->free_thr_log;
	M.hit = (float)m->hit_log;
	M.clamp_min = (float)m->cmin_log;
	M.clamp_max = (float)m->cmax_log;
	// toProb(float) with expf, as the reference evaluates it on the host
	M.prob_hit = 1.0 / (1.0 + (double)expf(-M.hit));
	// float thresholds exactly equivalent to the reference's double-vs-float compares
	{
		float fc = (float)m->free_thr_log;
		if ((double)fc < m->free_thr_log) fc = nextafterf(fc, INFINITY);
		float of = (float)m->occ_thr_log;
		if ((double)of > m->occ_thr_log) of = nextafterf(of, -INFINITY);
		M.free_ceil = fc;
		M.occ_floor = of;
	}
	uint32_t f = (m->free_thr_log > 0.0) ? 1u : 0u;
	if (m->free_thr_log <= 0.0 && m->occ_thr_log >= 0.0) f |= 2u;
	M.default_flags = f;
}

void reset_bbox(Map* m)
{
	double h = node_half(m->M.g, m->M.g.depth_levels);
	for (int i = 0; i < 3; ++i) {
		m->min_change[i] = h;
		m->max_change[i] = -h;
	}
}

// ---- brick and upper-node pools --------------------------------------------------------------
enum class Unit { kSlot, kBrick, kUpper };  // block slot (64 per brick), brick, upper node
// when an array exists: always, on colour maps, or from the first out-of-tree key (alias masks) /
// the first enableChangeDetection (change mask) on
enum class Exists { kAlways, kColour, kAlias, kChange };

struct PoolArray {
	Buffer<unsigned char>& buf;  // empty while the array does not exist
	Unit unit;
	size_t unit_bytes;  // bytes per unit
	int fill;           // byte the array (and every part added by a growth) starts as
	Exists exists;
	bool cleared;  // ufo_b200_clear resets the part in use
};

size_t capacity(const DeviceMap& M, Unit u)
{
	return u == Unit::kSlot ? (size_t)M.brick_cap * 64 : (u == Unit::kBrick ? M.brick_cap : M.up_cap);
}

size_t in_use(const Map* m, Unit u)
{
	return u == Unit::kSlot ? (size_t)m->n_bricks * 64 : (u == Unit::kBrick ? m->n_bricks : m->n_upper);
}

// Calls f(PoolArray) for every array of the two pools, then points the array's view (a DeviceMap
// field or a field of the map) at its buffer.  The hash tables and counters are sized on their own.
template <class F>
void for_each_pool_array(Map* m, F&& f)
{
	DeviceMap& M = m->M;
	size_t i = 0;
	auto array = [&](auto*& view, Unit unit, size_t per_unit, int fill, Exists exists, bool cleared) {
		using T = std::remove_reference_t<decltype(*view)>;
		if (i == m->pool.size()) m->pool.emplace_back(&m->device_bytes);
		Buffer<unsigned char>& buf = m->pool[i++];
		f(PoolArray{buf, unit, per_unit * sizeof(T), fill, exists, cleared});
		view = reinterpret_cast<T*>(buf.get());
	};
	const Unit S = Unit::kSlot, B = Unit::kBrick, U = Unit::kUpper;
	const Exists all = Exists::kAlways, colour = Exists::kColour;
	//    view              unit  per unit  fill  exists          cleared
	array(M.brick_key,      B,    1,        0,    all,            false);
	array(M.brick_stamp,    B,    1,        0,    all,            true);
	array(M.touched,        B,    1,        0,    all,            false);
	array(M.touched_alt,    B,    1,        0,    all,            false);
	array(M.touched_mi,     B,    1,        0,    all,            false);
	array(M.touched_alt_mi, B,    1,        0,    all,            false);
	array(M.brick_sum3,     B,    8,        0,    all,            false);
	array(M.brick_sum4,     B,    1,        0,    all,            false);
	array(M.brick_parent,   B,    1,        0xff, all,            true);
	array(M.brick_rgb3,     B,    8,        0,    colour,         false);
	array(M.brick_rgb4,     B,    1,        0,    colour,         false);
	array(M.leaf,           S,    64,       0,    all,            true);
	array(M.miss_mask,      S,    1,        0,    all,            true);
	array(M.hit_mask,       S,    1,        0,    all,            true);
	array(M.agg2,           S,    1,        0,    all,            true);
	array(M.meta,           S,    1,        0,    all,            true);
	array(M.sum1,           S,    8,        0,    all,            false);
	array(M.leaf_rgb,       S,    64,       0,    colour,         true);
	array(M.sum1_rgb,       S,    8,        0,    colour,         false);
	array(M.rgb2,           S,    1,        0,    colour,         false);
	array(M.alias_miss,     S,    1,        0,    Exists::kAlias, true);
	array(M.alias_hit,      S,    1,        0,    Exists::kAlias, true);
	array(m->chg_mask,      S,    1,        0,    Exists::kChange, true);
	array(M.up_key,         U,    1,        0,    all,            false);
	array(M.up_agg,         U,    1,        0,    all,            false);
	array(M.up_stamp,       U,    1,        0,    all,            true);
	array(M.up_child,       U,    8,        0,    all,            false);
	array(M.up_valid,       U,    1,        0,    all,            true);
	array(M.up_parent,      U,    1,        0xff, all,            true);
	array(M.up_rgb,         U,    1,        0,    colour,         false);
	array(M.up_child_rgb,   U,    8,        0,    colour,         false);
	array(m->d_list[0],     U,    1,        0,    all,            false);
	array(m->d_list[1],     U,    1,        0,    all,            false);
	// the kernels record changes while chg_mask is set
	M.chg_mask = m->chg_recording ? m->chg_mask : nullptr;
}

// allocates the arrays of one kind that do not exist yet, at the pools' capacities
void alloc_arrays(Map* m, Exists kind)
{
	for_each_pool_array(m, [&](const PoolArray& a) {
		if (a.exists == kind && !a.buf.get()) a.buf.resize(capacity(m->M, a.unit) * a.unit_bytes, a.fill, m->stream);
	});
}

// the hash tables: open addressing at a load of at most 1/2, contents not kept
void alloc_brick_hash(Map* m)
{
	DeviceMap& M = m->M;
	M.bh_mask = std::max(kMinHash, next_pow2(2ull * M.brick_cap)) - 1;
	m->bh_tab.resize((size_t)M.bh_mask + 1, 0xff, m->stream);
	M.bh_tab = m->bh_tab.get();
}

void alloc_upper_hash(Map* m)
{
	DeviceMap& M = m->M;
	M.uh_mask = std::max(kMinHash, next_pow2(2ull * M.up_cap)) - 1;
	m->uh_keys.resize((size_t)M.uh_mask + 1, 0xff, m->stream);
	m->uh_vals.resize((size_t)M.uh_mask + 1, 0xff, m->stream);
	M.uh_keys = m->uh_keys.get();
	M.uh_vals = m->uh_vals.get();
}

void alloc_pools(Map* m, uint32_t brick_cap, uint32_t up_cap)
{
	DeviceMap& M = m->M;
	M.brick_cap = brick_cap;
	M.up_cap = up_cap;
	alloc_brick_hash(m);
	alloc_upper_hash(m);
	alloc_arrays(m, Exists::kAlways);
	if (M.color) alloc_arrays(m, Exists::kColour);
	m->ctr.resize(1, 0, m->stream);
	M.ctr = m->ctr.get();
}

void push_counters(Map* m)
{
	// host view -> device allocation counters, clears the per-scan part
	Counters c{};
	c.n_blocks = m->n_blocks;
	c.n_bricks = m->n_bricks;
	c.n_upper = m->n_upper;
	for (int i = 0; i < 3; ++i) {
		c.bbox[i] = ~0ull;
		c.bbox[3 + i] = 0ull;
	}
	*m->h_ctr = c;
	CK(cudaMemcpyAsync(m->M.ctr, m->h_ctr.get(), sizeof(Counters), cudaMemcpyHostToDevice, m->stream));
}

// grows the existing arrays of the brick pools (upper = false) or of the upper-node pool to the
// capacities M holds now
void grow_arrays(Map* m, bool upper)
{
	for_each_pool_array(m, [&](const PoolArray& a) {
		if ((a.unit == Unit::kUpper) == upper && a.buf.get())
			a.buf.grow(capacity(m->M, a.unit) * a.unit_bytes, a.fill, m->stream);
	});
}

// grow whichever pool overflowed; `want_*` are the allocation counters the failed
// run reached (an over-estimate of the need)
void grow_pools(Map* m, uint32_t overflow, uint32_t want_bricks, uint32_t want_upper)
{
	DeviceMap& M = m->M;
	cudaStream_t s = m->stream;
	CK(cudaStreamSynchronize(s));
	if (overflow & 2u) {
		uint32_t oc = M.brick_cap;
		// marking stops creating bricks once the pool is exhausted, so `want` is barely above the old
		// capacity: small pools grow by 4x, large ones by 2x
		uint32_t nc = (uint32_t)std::max<uint64_t>((oc < (1u << 18) ? 4ull : 2ull) * oc, (uint64_t)want_bricks + want_bricks / 4);
		if ((uint64_t)nc * 64 > 0xfffffff0ull) throw std::bad_alloc();
		M.brick_cap = nc;
		grow_arrays(m, false);
		// rebuild the hash from the surviving bricks (drops kFailed entries)
		alloc_brick_hash(m);
		uint32_t live = std::min(m->h_ctr->n_bricks, oc);
		if (live) k_rebuild_brick_hash<<<(live + 255) / 256, 256, 0, s>>>(M, live);
		if (M.up_cap < nc / 2) overflow |= 4u;  // keep the upper-node pool in proportion
	}
	if (overflow & 4u) {
		uint32_t oc = M.up_cap;
		uint32_t nc = (uint32_t)std::max<uint64_t>(std::max<uint64_t>(2ull * oc, M.brick_cap / 2), (uint64_t)want_upper + want_upper / 4);
		M.up_cap = nc;
		grow_arrays(m, true);
		alloc_upper_hash(m);
		uint32_t nu = std::min(m->h_ctr->n_upper, oc);
		if (nu) k_rebuild_upper_hash<<<(nu + 255) / 256, 256, 0, s>>>(M, nu);
	}
	CK(cudaGetLastError());
}

size_t layout_stride(int layout)
{
	switch (layout) {
		case UFO_B200_XYZ_F64: return 24;
		case UFO_B200_XYZ_F32: return 12;
		case UFO_B200_XYZRGB_F64: return 32;
		case UFO_B200_XYZRGB_F32: return 16;
		default: return 0;
	}
}

// called with the stream idle
void ensure_scan_buffers(Map* m, size_t n, bool need_table, bool records, bool fused)
{
	cudaStream_t s = m->stream;
	if (n > m->d_hit_tab.size()) {
		m->d_seg_base.reset();  // sized by the ray capacity: allocated again below when needed
		m->d_seg_count.reset();
		m->d_order.reset();
		const size_t cap = std::max<size_t>(n, 1024);
		m->d_ray_end.resize(cap * 3, 0, s);
		m->d_hit_tab.resize(cap, 0xff, s);
	}
	const size_t ray_cap = m->d_hit_tab.size();
	if (records && !m->d_seg_base.get()) {
		m->d_seg_base.resize(ray_cap / 32 + 1, 0, s);
		m->d_seg_count.resize(ray_cap / 32 + 1, 0, s);
		m->d_order.resize(ray_cap / 32 + 1, 0, s);
	}
	if (fused && m->d_rc.size() < ray_cap) {
		m->d_items.resize(ray_cap * kShells);  // written before read
		m->d_vmask.resize((ray_cap / 32 + 1) * kShells, 0, s);
		m->d_rc.resize(ray_cap, 0, s);
	}
	if (need_table) {
		uint32_t want = std::max(1u << 12, next_pow2(4ull * n));
		if (want > m->d_tab_keys.size()) {
			m->d_tab_keys.resize(want, 0xff, s);
			m->d_tab_min.resize(want, 0xff, s);
		}
	}
}

void finish_stats(Map* m)
{
	// called after the stream is idle and h_ctr holds the end-of-scan counters
	if (!m->stats_pending) return;
	const Counters& c = *m->h_ctr;
	ufo_b200_scan_stats& st = m->stats;
	unsigned long long sum[8] = {0, 0, 0, 0, 0, 0, 0, 0};
	for (int sl = 0; sl < kStatSlots; ++sl)
		for (int k = 0; k < 8; ++k) sum[k] += c.stat[sl][k];
	st.rays = c.n_rays;
	st.visits = c.visits;
	st.touched_voxels = sum[0];
	st.hit_voxels = sum[1];
	st.touched_octets = sum[2];
	st.touched_blocks = sum[3];
	st.touched_d3 = sum[6];
	st.touched_bricks = sum[5];
	st.touched_lines = sum[7];
	st.upper_nodes = c.upper_nodes;
	m->n_blocks += (uint32_t)sum[4];
	m->n_bricks = std::min(c.n_bricks, m->M.brick_cap);
	m->n_upper = std::min(c.n_upper, m->M.up_cap);
	st.blocks_in_map = m->n_blocks;
	st.bricks_in_map = m->n_bricks;
	st.device_bytes = m->device_bytes;
	if (c.n_rays || sum[0]) {
		for (int i = 0; i < 3; ++i) {
			if (c.bbox[i] != ~0ull) m->min_change[i] = std::min(m->min_change[i], decode_ordered(c.bbox[i]));
			if (c.bbox[3 + i] != 0ull)
				m->max_change[i] = std::max(m->max_change[i], decode_ordered(c.bbox[3 + i]));
		}
	}
	if (m->ev_valid) {
		cudaEventElapsedTime(&st.ms_total, m->ev[0], m->ev[6]);
		if (m->h2d_valid) cudaEventElapsedTime(&st.ms_h2d, m->ev_copy0, m->ev_copied);
		if (m->profiling) {
			cudaEventElapsedTime(&st.ms_points, m->ev[0], m->ev[2]);
			if (m->ev7_valid) {
				cudaEventElapsedTime(&st.ms_rays, m->ev[2], m->ev[7]);
				cudaEventElapsedTime(&st.ms_scatter, m->ev[7], m->ev[3]);
			} else {
				cudaEventElapsedTime(&st.ms_rays, m->ev[2], m->ev[3]);
			}
			cudaEventElapsedTime(&st.ms_update, m->ev[3], m->ev[5]);
			cudaEventElapsedTime(&st.ms_propagate, m->ev[5], m->ev[6]);
		}
	}
	m->stats_pending = false;
}

void ensure_seg(Map* m, unsigned long long want)
{
	if (want <= m->d_seg.size()) return;
	CK(cudaStreamSynchronize(m->stream));
	m->d_seg.resize(want);
}

// K3 over the scan's touched list: persistent warps, the list length is read on the device.
void launch_update(Map* m, float miss, bool set_mode = false)
{
	if (m->M.color) {
		const uint32_t per_sm = UbShape<true>::kMinBlocks, T = UbShape<true>::kWarps * 32;
		const uint32_t grid = (uint32_t)m->sm_count * (m->k3_blocks ? std::min<uint32_t>(per_sm, (uint32_t)m->k3_blocks) : per_sm);
		if (set_mode) k_update_brick<true, true><<<grid, T, 0, m->stream>>>(m->M, miss);
		else k_update_brick<true, false><<<grid, T, 0, m->stream>>>(m->M, miss);
	} else {
		const uint32_t per_sm = UbShape<false>::kMinBlocks, T = UbShape<false>::kWarps * 32;
		const uint32_t grid = (uint32_t)m->sm_count * (m->k3_blocks ? std::min<uint32_t>(per_sm, (uint32_t)m->k3_blocks) : per_sm);
		if (set_mode) k_update_brick<false, true><<<grid, T, 0, m->stream>>>(m->M, miss);
		else k_update_brick<false, false><<<grid, T, 0, m->stream>>>(m->M, miss);
	}
	++m->launches;
}

// generic marking path: walk -> (block, mask) records -> k_scatter.  Handles every insert depth,
// out-of-tree keys and the fixed-step variant.
void launch_rays_records(Map* m, const ScanArgs& a, int simple)
{
	if (simple) {
		k_rays_simple<<<(a.n + 127) / 128, 128, 0, m->stream>>>(m->M, a);
		++m->launches;
		if (a.depth >= 5) {
			k_expand_nodes<<<m->sm_count * 8, 256, 0, m->stream>>>(m->M, a);
			++m->launches;
		}
		return;
	}
	// one resident wave; batches are ordered by work and dealt round-robin over the CTAs
	uint32_t* counter = &m->M.ctr->ray_batch;
	uint32_t n_batches = (a.n + 31) / 32;
	k_order_batches<<<1, 1024, 0, m->stream>>>(a.seg_count, n_batches, a.order);
	++m->launches;
	uint32_t need = (a.n + kRayThreads - 1) / kRayThreads;
	uint32_t grid = std::min<uint32_t>(need, (uint32_t)m->sm_count * m->ray_blocks_per_sm);
	if (a.count_visits) {
		if (a.depth == 0) k_rays<0, true><<<grid, kRayThreads, 0, m->stream>>>(m->M, a, counter);
		else if (a.depth == 1) k_rays<1, true><<<grid, kRayThreads, 0, m->stream>>>(m->M, a, counter);
		else k_rays<2, true><<<grid, kRayThreads, 0, m->stream>>>(m->M, a, counter);
	} else {
		if (a.depth == 0) k_rays<0, false><<<grid, kRayThreads, 0, m->stream>>>(m->M, a, counter);
		else if (a.depth == 1) k_rays<1, false><<<grid, kRayThreads, 0, m->stream>>>(m->M, a, counter);
		else k_rays<2, false><<<grid, kRayThreads, 0, m->stream>>>(m->M, a, counter);
	}
	++m->launches;
	if (m->profiling) {
		CK(cudaEventRecord(m->ev[7], m->stream));
		m->ev7_valid = true;
	}
	{
		// all CTAs resident, looping over the work items (j, region) with stride = grid size.
		// The grid size is made coprime with the number of regions so that every CTA walks
		// through ALL regions: region length correlates with the region index (ring order of
		// the sensor), and a stride sharing a factor with it gives some CTAs only long regions.
		uint32_t sgrid = (uint32_t)m->sm_count * 8;
		const uint32_t n_regions = (a.n + 31) / 32;
		while (sgrid > 1 && std::gcd(sgrid, n_regions) != 1) --sgrid;
		const bool generic = a.depth >= 3 || m->M.alias_miss, shard = m->M.shard_world > 1;
		if (generic && shard) k_scatter<true, true><<<sgrid, kChunk, 0, m->stream>>>(m->M, a);
		else if (generic) k_scatter<true, false><<<sgrid, kChunk, 0, m->stream>>>(m->M, a);
		else if (shard) k_scatter<false, true><<<sgrid, kChunk, 0, m->stream>>>(m->M, a);
		else k_scatter<false, false><<<sgrid, kChunk, 0, m->stream>>>(m->M, a);
	}
	++m->launches;
	if (a.depth >= 5) {
		k_expand_nodes<<<m->sm_count * 8, 256, 0, m->stream>>>(m->M, a);
		++m->launches;
	}
}

template <int DEPTH, bool DENSE>
void launch_fused_depth(Map* m, const ScanArgs& a)
{
	cudaStream_t s = m->stream;
	const uint32_t n_batches = (a.n + 31) / 32;
	const uint32_t sgrid = (n_batches * 32 + 127) / 128;
	if (a.count_visits) k_split<DEPTH, true><<<sgrid, 128, 0, s>>>(m->M, a);
	else k_split<DEPTH, false><<<sgrid, 128, 0, s>>>(m->M, a);
	const uint32_t grid = (uint32_t)m->sm_count * m->walk_blocks_per_sm;
	const bool shard = m->M.shard_world > 1 && !DENSE;  // dense: ownership is applied by k_gather
	if (a.count_visits) {
		if (shard) k_walk_mark<DEPTH, true, true, DENSE><<<grid, kWalkThreads, 0, s>>>(m->M, a);
		else k_walk_mark<DEPTH, false, true, DENSE><<<grid, kWalkThreads, 0, s>>>(m->M, a);
	} else {
		if (shard) k_walk_mark<DEPTH, true, false, DENSE><<<grid, kWalkThreads, 0, s>>>(m->M, a);
		else k_walk_mark<DEPTH, false, false, DENSE><<<grid, kWalkThreads, 0, s>>>(m->M, a);
	}
	m->launches += 2;
	if (DENSE) {
		if (m->profiling) {
			CK(cudaEventRecord(m->ev[7], s));
			m->ev7_valid = true;
		}
		k_gather_scan<<<m->sm_count * 2, 256, 0, s>>>(m->M);
		if (m->M.shard_world > 1) k_gather<true><<<m->sm_count * 8, 256, 0, s>>>(m->M);
		else k_gather<false><<<m->sm_count * 8, 256, 0, s>>>(m->M);
		m->launches += 2;
	}
}

// fused path (ufo_walk.cuh): insert depth <= 2, no out-of-tree keys seen by this map
void launch_rays_fused(Map* m, const ScanArgs& a)
{
	if (m->M.dense) {
		if (a.depth == 0) launch_fused_depth<0, true>(m, a);
		else if (a.depth == 1) launch_fused_depth<1, true>(m, a);
		else launch_fused_depth<2, true>(m, a);
	} else {
		if (a.depth == 0) launch_fused_depth<0, false>(m, a);
		else if (a.depth == 1) launch_fused_depth<1, false>(m, a);
		else launch_fused_depth<2, false>(m, a);
	}
}

bool use_fused(const Map* m, const PendingScan& p)
{
	return !p.has_vol && !p.simple && p.a.depth <= 2 && !m->M.alias_miss && !m->force_records;
}

// Dense scan volume: bricks per axis a scan of this range needs around the sensor (0: no volume)
uint32_t volume_bricks(const Map* m, const PendingScan& p)
{
	if (m->no_dense || !(p.a.max_range > 0)) return 0;
	const double vox = p.a.max_range * m->M.g.resolution_factor + 4.0;  // ray length in voxels + slack
	if (vox > 16.0 * 160) return 0;  // > 320 bricks per axis (16.8 GB of masks): use the hash path
	const uint32_t half = (uint32_t)(vox / 16.0) + 2;
	return 2 * half + 1;
}

// called with the stream idle; binds the volume to this scan's sensor position
void setup_volume(Map* m, PendingScan& p, uint32_t db)
{
	DeviceMap& M = m->M;
	if (db > m->vol_db_cap) {
		const size_t nb = (size_t)db * db * db;
		m->vol.resize(nb * 64, 0, m->stream);
		m->vol_dirty.resize(nb / 64 + 1, 0, m->stream);
		m->vol_list.resize(nb / 64 + 1, 0, m->stream);
		M.vol = m->vol.get();
		M.vol_dirty = m->vol_dirty.get();
		M.vol_list = m->vol_list.get();
		m->vol_db_cap = db;
	}
	const Geometry& g = M.g;
	const uint32_t half = (db - 1) / 2;
	const Key3 ko = point_to_key(g, p.a.origin, 0);
	M.vol_db = db;
	M.vol_g0x = ((ko.x & 0x1fffffu) >> 4) - half;
	M.vol_g0y = ((ko.y & 0x1fffffu) >> 4) - half;
	M.vol_g0z = ((ko.z & 0x1fffffu) >> 4) - half;
}

// drops the marks left in the scan volume
void wipe_volume(Map* m)
{
	m->vol.fill(0, m->stream);
	m->vol_dirty.fill(0, m->stream);
}

// K4: upper levels, depth 5 .. L, from the touched list
void launch_upper_seed(Map* m)
{
	DeviceMap& M = m->M;
	if (M.g.depth_levels < 5) return;
	// list_count[] is zero when the first seed of a pass runs; level d reads list d&1 ? 0 : 1
	k_upper_seed<<<m->sm_count * 2, 256, 0, m->stream>>>(M, m->d_list[0], M.up_cap);
	++m->launches;
}

void launch_upper_levels(Map* m)
{
	DeviceMap& M = m->M;
	cudaStream_t s = m->stream;
	if (M.g.depth_levels < 5) return;
	const uint32_t L = M.g.depth_levels;
	for (uint32_t d = 5; d <= std::min(6u, L); ++d) {
		k_upper_level<<<m->sm_count, 256, 0, s>>>(M, d, m->d_list[(d & 1) ? 0 : 1], m->d_list[(d & 1) ? 1 : 0], M.up_cap);
		++m->launches;
	}
	if (L >= 7) {
		k_upper_tail<<<1, 1024, 0, s>>>(M, 7, m->d_list[0], m->d_list[1], M.up_cap);
		++m->launches;
	}
	CK(cudaGetLastError());
}

void launch_upper(Map* m)
{
	launch_upper_seed(m);
	launch_upper_levels(m);
}

__global__ void k_reset_upper_pass(Counters* c, uint32_t n_upper)
{
	c->overflow = 0;
	c->list_count[0] = c->list_count[1] = c->list_count[2] = 0;
	c->upper_nodes = 0;
	c->n_upper = n_upper;
}

// Enqueues every kernel of one scan and the read-back of its counters; never waits.
void enqueue_scan(Map* m, PendingScan& p)
{
	DeviceMap& M = m->M;
	cudaStream_t s = m->stream;
	ScanArgs& a = p.a;
	M.scan_id++;
	if (M.scan_id == 0) M.scan_id = 1;
	M.up_epoch++;
	if (M.up_epoch == 0) M.up_epoch = 1;
	const bool fused = use_fused(m, p);
	M.dense = (fused && p.dense) ? 1u : 0u;
	M.mask_base = M.dense ? M.vol : M.miss_mask;
	// (re-)bind the scan buffers: they may have been regrown since the scan was first enqueued
	a.ray_end = m->d_ray_end.get();
	a.tab_keys = m->d_tab_keys.get();
	a.tab_min = m->d_tab_min.get();
	a.tab_mask = m->d_tab_keys.size() ? (uint32_t)m->d_tab_keys.size() - 1 : 0;
	a.hit_tab = p.use_color ? m->d_hit_tab.get() : nullptr;
	a.seg = nullptr;
	a.seg_base = a.seg_count = a.order = nullptr;
	a.items = nullptr;
	if (fused) {
		a.items = m->d_items.get();
		a.item_stride = m->d_rc.size();
		a.vmask = m->d_vmask.get();
		a.rc = m->d_rc.get();
	} else if (!p.simple && !p.has_vol) {
		a.seg = m->d_seg.get();
		a.seg_cap = m->d_seg.size();
		a.seg_base = m->d_seg_base.get();
		a.seg_count = m->d_seg_count.get();
		a.order = m->d_order.get();
	}
	if (a.depth >= 5) {
		if (!m->d_nodes.get()) m->d_nodes.resize((size_t)1 << 20, 0, s);
		a.nodes = m->d_nodes.get();
		a.nodes_cap = 1u << 20;
	}
	m->ev7_valid = false;
	push_counters(m);
	if (p.need_table) {
		m->d_tab_keys.fill(0xff, s);
		m->d_tab_min.fill(0xff, s);
	}
	if (p.has_vol) {
		// setValueVolume: the marks come from the box instead of a scan
		k_volume_mark<<<p.vol.nx * p.vol.ny * p.vol.nz, 64, 0, s>>>(M, p.vol);
		++m->launches;
		if (m->profiling) CK(cudaEventRecord(m->ev[2], s));
	} else if (a.n) {
		uint32_t grid = (uint32_t)((a.n + 255) / 256);
		k_points<<<grid, 256, 0, s>>>(M, a);
		++m->launches;
		if (p.use_color) {
			k_hits<<<grid, 256, 0, s>>>(M, a);
			++m->launches;
		}
		if (m->profiling) CK(cudaEventRecord(m->ev[2], s));
		if (fused) launch_rays_fused(m, a);
		else launch_rays_records(m, a, p.simple);
	} else if (m->profiling) {
		CK(cudaEventRecord(m->ev[2], s));
	}
	if (m->profiling) CK(cudaEventRecord(m->ev[3], s));
	CK(cudaGetLastError());
	// K3 and K4 run off the device-side touched list; if a pool overflowed while marking they
	// back off by themselves and the scan is repeated by finalize_scan() after the growth.
	const bool aliases = M.alias_miss != nullptr;
	const uint32_t agrid = (uint32_t)m->sm_count * 4;
	if (aliases) {
		k_alias_apply<<<agrid, 256, 0, s>>>(M, M.hit, 1);
		++m->launches;
	}
	launch_update(m, p.has_vol ? p.set_value : a.miss, p.has_vol);
	if (aliases) {
		k_alias_apply<<<agrid, 256, 0, s>>>(M, a.miss, 0);
		k_alias_refresh<<<agrid, 256, 0, s>>>(M);
		if (M.color) k_brick_agg<true><<<agrid, 256, 0, s>>>(M);
		else k_brick_agg<false><<<agrid, 256, 0, s>>>(M);
		m->launches += 3;
	}
	if (m->profiling) CK(cudaEventRecord(m->ev[5], s));
	launch_upper(m);
	CK(cudaEventRecord(m->ev[6], s));
	m->ev_valid = true;
	CK(cudaMemcpyAsync(m->h_ctr.get(), M.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
	m->stats_pending = true;
	p.valid = true;
}

// Waits for the scan in flight, repeats it if a device pool overflowed, and folds its counters
// into the host view.  Throws MapError if the scan cannot be completed.
void finalize_scan(Map* m)
{
	CK(cudaStreamSynchronize(m->stream));
	PendingScan& p = m->pending;
	if (!p.valid) {
		finish_stats(m);
		return;
	}
	DeviceMap& M = m->M;
	if (p.routed) {
		const uint32_t rf = m->h_route_flag.get() ? *m->h_route_flag : 0u;
		if (rf || (m->route_stage == 1 && m->h_ctr->overflow)) {
			if (rf) m->set_error("routed mode: an inbox region is too small (flags %u); raise cap_bricks / cap_hits", rf);
			else m->set_error("routed mode: a device pool overflowed while marking (flags %u); create the map with a larger initial_bricks", m->h_ctr->overflow);
			p.valid = false;
			m->stats_pending = false;
			m->poisoned = true;
			m->route_stage = 0;
			throw MapError{UFO_B200_E_NOMEM};
		}
		if (m->route_stage == 1) return;  // marked, not applied yet: nothing to fold in
	}
	while (true) {
		const uint32_t ov = m->h_ctr->overflow;
		if (!ov) break;
		++p.regrows;
		if (p.regrows > 16 || (ov & (16u | 128u)) || p.routed) {
			if (ov & 128u) m->set_error("insert depth >= 5 with rays that leave the map (out-of-tree nodes) is not supported");
			else if (ov & 16u) m->set_error("internal error: a ray walk exceeded its record bound");
			else if (p.routed) m->set_error("routed mode: a device pool overflowed (flags %u); create the map with a larger initial_bricks", ov);
			else m->set_error("device pools keep overflowing");
			p.valid = false;
			m->stats_pending = false;
			m->poisoned = true;  // marks of the failed scan are still in the masks
			throw MapError{(ov & 128u) ? UFO_B200_E_UNSUPPORTED : ((ov & 16u) ? UFO_B200_E_CUDA : UFO_B200_E_NOMEM)};
		}
		try {
			if (ov == 4u) {
				// only the upper-node pool overflowed: the leaves are updated, repeat the propagation
				const uint32_t nu = std::min(m->h_ctr->n_upper, M.up_cap);
				grow_pools(m, 4u, 0, m->h_ctr->n_upper);
				M.up_epoch++;
				k_reset_upper_pass<<<1, 1, 0, m->stream>>>(M.ctr, nu);
				launch_upper(m);
				CK(cudaEventRecord(m->ev[6], m->stream));
				CK(cudaMemcpyAsync(m->h_ctr.get(), M.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, m->stream));
			} else {
				// an allocation failed while marking: nothing was consumed (K3/K4 backed off).  Grow,
				// keep the bricks that were created, and run the whole scan again under a new scan id
				// (marking is idempotent: OR into masks, find-or-create of bricks).
				m->n_bricks = std::min(m->h_ctr->n_bricks, M.brick_cap);
				if (ov & 64u) {
					// a mark fell outside the scan volume (cannot happen for rays within max_range; kept
					// as a safety net): wipe the volume and repeat through the brick hash
					m->no_dense = 1;
					p.dense = false;
					wipe_volume(m);
				}
				if (ov & 32u) {
					// first out-of-tree key ever seen by this map: allocate the alias mask arrays;
					// from now on this map uses the generic record path
					alloc_arrays(m, Exists::kAlias);
					if (p.dense) {
						// the marks the walk already left in the volume are not consumed by the record path
						wipe_volume(m);
						p.dense = false;
					}
				}
				const bool fused = use_fused(m, p);
				if (!fused && !p.simple && !p.has_vol) {
					ensure_scan_buffers(m, p.a.n, false, true, false);
					unsigned long long want = std::max<unsigned long long>(m->h_ctr->seg_total + m->h_ctr->seg_total / 4 + 1024,
					                                                        std::max<unsigned long long>(p.a.n, 1024) * 48ull);
					ensure_seg(m, want);
				}
				if (ov & 6u) grow_pools(m, ov & 6u, m->h_ctr->n_bricks, m->h_ctr->n_upper);
				enqueue_scan(m, p);
			}
		} catch (std::bad_alloc&) {
			m->set_error("block pool cannot grow beyond 2^32 slots");
			p.valid = false;
			m->stats_pending = false;
			m->poisoned = true;
			throw MapError{UFO_B200_E_NOMEM};
		}
		CK(cudaStreamSynchronize(m->stream));
	}
	m->stats.regrows = p.regrows;
	m->stats.launches = m->launches;
	m->stats.result_bytes = sizeof(Counters) * (1 + p.regrows);
	p.valid = false;
	finish_stats(m);
	m->done_stats = m->stats;
}

// every brick of the map becomes the "touched list" (whole-map passes: threshold changes)
__global__ void k_touch_all(DeviceMap M, uint32_t n_bricks)
{
	for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < n_bricks; b += gridDim.x * blockDim.x) {
		M.touched[b] = b;
		M.brick_stamp[b] = M.scan_id;
	}
	if (blockIdx.x == 0 && threadIdx.x == 0) M.ctr->n_touched = n_bricks;
}

// contains_free / contains_unknown of depth 1 and 2 from the leaves, under the current thresholds
__global__ void __launch_bounds__(256) k_reflag(DeviceMap M, uint32_t n_bricks)
{
	const size_t n = (size_t)n_bricks * 64;
	for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < n; b += (size_t)gridDim.x * blockDim.x) {
		const uint32_t mt = M.meta[b];
		if (!(mt & 0xff0000u)) continue;
		const float* leaf = M.leaf + b * 64;
		uint32_t bfl = 0, fl16 = 0;
		for (uint32_t o = 0; o < 8; ++o) {
			uint32_t ofl = M.default_flags;
			if ((mt >> (16 + o)) & 1u) {
				ofl = 0;
				for (int j = 0; j < 8; ++j) ofl |= leaf_flags(M, leaf[8 * o + j]);
				fl16 |= ofl << (2 * o);
			}
			bfl |= ofl;
		}
		M.meta[b] = (mt & 0xffff0000u) | fl16;
		M.agg2[b].flags = bfl;
	}
}

// The reference re-reads the whole tree when the occupied / free thresholds change
// (setOccupiedFreeThres, occupancy_map_base.h:748-761): the contains_free / contains_unknown
// flags of every inner node are functions of the thresholds.  Same effect here.
void rebuild_flags(Map* m)
{
	finalize_scan(m);
	if (!m->n_bricks) return;
	DeviceMap& M = m->M;
	cudaStream_t s = m->stream;
	M.scan_id++;
	if (M.scan_id == 0) M.scan_id = 1;
	M.up_epoch++;
	push_counters(m);
	k_touch_all<<<m->sm_count, 256, 0, s>>>(M, m->n_bricks);
	k_reflag<<<m->sm_count * 8, 256, 0, s>>>(M, m->n_bricks);
	if (M.color) k_brick_agg<true><<<m->sm_count * 4, 256, 0, s>>>(M);
	else k_brick_agg<false><<<m->sm_count * 4, 256, 0, s>>>(M);
	launch_upper(m);
	CK(cudaStreamSynchronize(s));
}

int sync_map(Map* m)
{
	finalize_scan(m);
	return UFO_B200_OK;
}

// Starts the copy of a host cloud to the device, on the copy stream, into the staging buffer the
// scan in flight is not using: the H2D copy of scan k+1 overlaps the kernels of scan k (the
// reference overlaps its own front end with the previous scan's helper thread the same way,
// OMB:315).  Returns where the scan reads the points.
const void* stage_points(Map* m, const void* points, size_t bytes)
{
	m->stage ^= 1u;
	Buffer<unsigned char>& buf = m->d_points[m->stage];
	if (bytes > buf.size()) buf.resize(std::max<size_t>(bytes + bytes / 8, 1 << 16));
	CK(cudaEventRecord(m->ev_copy0, m->copy_stream));
	CK(cudaMemcpyAsync(buf.get(), points, bytes, cudaMemcpyHostToDevice, m->copy_stream));
	CK(cudaEventRecord(m->ev_copied, m->copy_stream));
	return buf.get();
}

int do_insert(Map* m, const double origin[3], const void* points, bool on_device, size_t n,
              const double* frame_pose,
              int layout, double max_range, uint32_t depth, int simple, uint32_t early_stopping,
              int discrete, int async, const ufo_b200_cloud2* pc2 = nullptr, const VolumeArgs* vol = nullptr,
              float set_value = 0.0f)
{
	if (!m || !origin || (!points && n)) return UFO_B200_E_INVALID;
	size_t stride = pc2 ? pc2->point_step : layout_stride(layout);
	if (!stride || n > 0x7fffffffull) {
		m->set_error("invalid layout %d or point count %zu", layout, n);
		return UFO_B200_E_INVALID;
	}
	bool pc2_rgb = false;
	if (pc2) {
		layout = 4;
		pc2_rgb = pc2->off_r >= 0 && pc2->off_g >= 0 && pc2->off_b >= 0;
		const uint32_t fx[3] = {pc2->off_x, pc2->off_y, pc2->off_z};
		bool ok = pc2->point_step % 4 == 0;
		for (uint32_t f : fx) ok = ok && f % 4 == 0 && (size_t)f + 4 <= pc2->point_step;
		const int32_t fc[3] = {pc2->off_r, pc2->off_g, pc2->off_b};
		for (int32_t c : fc) ok = ok && (c < 0 || (size_t)c < pc2->point_step);
		if (!ok) {
			m->set_error("PointCloud2 descriptor: x/y/z must be 4-byte aligned FLOAT32 fields inside point_step");
			return UFO_B200_E_INVALID;
		}
	}
	if (early_stopping != 0) {
		m->set_error("early_stopping is order-dependent in the reference (occupancy_map_base.h:1289-1298) and is not supported");
		return UFO_B200_E_UNSUPPORTED;
	}
	if (depth > 6) {
		m->set_error("insert depth %u > 6 is not supported (a free-space node of depth 7 covers 512 bricks of the dense value field)", depth);
		return UFO_B200_E_UNSUPPORTED;
	}
	if (m->poisoned) {
		m->set_error("an earlier scan failed half-way; ufo_b200_clear() the map before inserting again");
		return UFO_B200_E_INVALID;
	}
	CK(cudaSetDevice(m->device));

	// an on-device cloud is read in place: it has to stay valid until the scan is done
	const size_t bytes = n * stride;
	const bool copied = !on_device && bytes;
	const void* src = copied ? stage_points(m, points, bytes) : points;
	// one integration in flight at most (insertPointCloudWait, occupancy_map_base.h:315)
	finalize_scan(m);

	DeviceMap& M = m->M;
	cudaStream_t s = m->stream;
	const bool has_rgb = layout == UFO_B200_XYZRGB_F64 || layout == UFO_B200_XYZRGB_F32 || pc2_rgb;
	PendingScan& p = m->pending;
	p = PendingScan{};
	p.use_color = M.color && has_rgb;
	p.need_table = discrete || p.use_color || depth >= 5;  // depth 5/6: the scan's set of free-space nodes
	p.simple = simple != 0;
	p.has_vol = vol != nullptr;
	if (vol) p.vol = *vol;
	p.set_value = set_value;

	ScanArgs& a = p.a;
	a.origin = {origin[0], origin[1], origin[2]};
	a.max_range = max_range;
	a.n = (uint32_t)n;
	a.depth = depth;
	a.layout = layout;
	a.discrete = discrete;
	a.use_color = p.use_color;
	a.miss = (float)(m->miss_log / (double)((2.0 * depth) + 1));
	a.count_visits = m->profiling >= 2;
	if (pc2) {
		a.pc2_step = pc2->point_step;
		a.pc2_x = pc2->off_x;
		a.pc2_y = pc2->off_y;
		a.pc2_z = pc2->off_z;
		a.pc2_r = pc2_rgb ? pc2->off_r : -1;
		a.pc2_g = pc2_rgb ? pc2->off_g : -1;
		a.pc2_b = pc2_rgb ? pc2->off_b : -1;
	}
	if (frame_pose) {
		a.has_frame = 1;
		a.frame = Frame{frame_pose[3], frame_pose[4], frame_pose[5], frame_pose[6],
		                frame_pose[0], frame_pose[1], frame_pose[2]};
	}
	const bool fused = use_fused(m, p);
	const bool records = !fused && !p.simple && !p.has_vol;
	ensure_scan_buffers(m, n, p.need_table, records, fused);
	if (fused) {
		const uint32_t db = volume_bricks(m, p);
		p.dense = db != 0;
		if (p.dense) setup_volume(m, p, db);
	}
	if (records) {
		// first guess for the record buffer: 48 records per ray; grown on demand
		ensure_seg(m, std::max<unsigned long long>(m->d_seg.size(), std::max<unsigned long long>(n, 1024) * 48ull));
	}
	a.points = src;

	m->stats = ufo_b200_scan_stats{};
	m->stats.points = n;
	m->launches = 0;
	m->h2d_valid = copied;
	CK(cudaEventRecord(m->ev[0], s));
	if (copied) CK(cudaStreamWaitEvent(s, m->ev_copied, 0));
	enqueue_scan(m, p);
	// the caller's buffer is free again when this returns (the reference takes the cloud by value)
	if (copied) CK(cudaEventSynchronize(m->ev_copied));
	if (!async) return sync_map(m);
	return UFO_B200_OK;
}

// ---- routed multi-GPU mode (ufo_route.cuh) -------------------------------------------------
size_t route_layout(uint32_t world, uint32_t cap_m, uint32_t cap_h, size_t* region, size_t* miss_off, size_t* hit_off)
{
	const size_t mo = 256;
	const size_t ho = mo + (((size_t)cap_m * kMissRecWords * 8 + 255) & ~(size_t)255);
	const size_t reg = ho + (((size_t)cap_h * 8 + 255) & ~(size_t)255);
	if (region) *region = reg;
	if (miss_off) *miss_off = mo;
	if (hit_off) *hit_off = ho;
	return reg * world * 2;
}

void route_fill_table(Map* m)
{
	RouteTable& T = *m->h_route;
	memset(&T, 0, sizeof(T));
	T.cap_m = m->route_cap_m;
	T.cap_h = m->route_cap_h;
	const uint32_t W = m->M.route_world, me = m->M.route_rank;
	for (uint32_t r = 0; r < W; ++r) {
		// my records for rank r land in r's inbox, region (parity, source = me)
		unsigned char* bo = static_cast<unsigned char*>(m->route_peer[r]) + ((size_t)m->route_parity * W + me) * m->route_region;
		T.out[r].hdr = reinterpret_cast<uint32_t*>(bo);
		T.out[r].miss = reinterpret_cast<unsigned long long*>(bo + m->route_miss_off);
		T.out[r].hit = reinterpret_cast<unsigned long long*>(bo + m->route_hit_off);
		unsigned char* bi = m->route_inbox.get() + ((size_t)m->route_parity * W + r) * m->route_region;
		T.in[r].hdr = reinterpret_cast<uint32_t*>(bi);
		T.in[r].miss = reinterpret_cast<unsigned long long*>(bi + m->route_miss_off);
		T.in[r].hit = reinterpret_cast<unsigned long long*>(bi + m->route_hit_off);
	}
}

int do_route_mark(Map* m, const double origin[3], const void* points, bool on_device, size_t n, int layout,
                  double max_range, int self_too)
{
	if (!m || !origin || (!points && n)) return UFO_B200_E_INVALID;
	const size_t stride = layout_stride(layout);
	if (!stride || n > 0x7fffffffull) return UFO_B200_E_INVALID;
	DeviceMap& M = m->M;
	if (M.route_world < 2 || !m->route_peer[0]) {
		m->set_error("routed mode is not set up (ufo_b200_route_setup + ufo_b200_route_connect)");
		return UFO_B200_E_INVALID;
	}
	if (M.color || M.alias_miss || m->poisoned || m->route_stage == 1) {
		m->set_error(m->route_stage == 1 ? "ufo_b200_route_mark: the previous pass was not applied"
		                                 : "routed mode needs a healthy mono map without out-of-tree keys");
		return UFO_B200_E_UNSUPPORTED;
	}
	CK(cudaSetDevice(m->device));
	const size_t bytes = n * stride;
	const bool copied = !on_device && bytes;
	const void* src = copied ? stage_points(m, points, bytes) : points;
	finalize_scan(m);
	cudaStream_t s = m->stream;
	PendingScan& p = m->pending;
	p = PendingScan{};
	p.routed = true;
	ScanArgs& a = p.a;
	a.origin = {origin[0], origin[1], origin[2]};
	a.max_range = max_range;
	a.n = (uint32_t)n;
	a.layout = layout;
	a.miss = (float)m->miss_log;
	a.count_visits = m->profiling >= 2;
	ensure_scan_buffers(m, n, false, false, true);
	{
		const uint32_t db = volume_bricks(m, p);
		p.dense = db != 0;
		if (p.dense) setup_volume(m, p, db);
	}
	M.dense = p.dense ? 1u : 0u;
	M.mask_base = M.dense ? M.vol : M.miss_mask;
	a.points = src;
	a.ray_end = m->d_ray_end.get();
	a.items = m->d_items.get();
	a.item_stride = m->d_rc.size();
	a.vmask = m->d_vmask.get();
	a.rc = m->d_rc.get();
	m->stats = ufo_b200_scan_stats{};
	m->stats.points = n;
	m->launches = 0;
	m->h2d_valid = copied;
	m->ev7_valid = false;
	M.route_self = self_too ? 1u : 0u;
	m->route_parity ^= 1u;
	route_fill_table(m);
	*m->h_route_flag = 0;
	CK(cudaEventRecord(m->ev[0], s));
	CK(cudaMemcpyAsync(M.route, m->h_route.get(), sizeof(RouteTable), cudaMemcpyHostToDevice, s));
	if (copied) CK(cudaStreamWaitEvent(s, m->ev_copied, 0));
	M.scan_id += 1;
	if (M.scan_id == 0) M.scan_id = 1;
	push_counters(m);
	if (n) {
		k_points<<<(uint32_t)((n + 255) / 256), 256, 0, s>>>(M, a);
		++m->launches;
		if (m->profiling) CK(cudaEventRecord(m->ev[2], s));
		launch_rays_fused(m, a);
	} else if (m->profiling) {
		CK(cudaEventRecord(m->ev[2], s));
	}
	k_outbox<<<m->sm_count * 4, 256, 0, s>>>(M);
	k_outbox_publish<<<1, 32, 0, s>>>(M);
	m->launches += 2;
	if (m->profiling) CK(cudaEventRecord(m->ev[3], s));
	CK(cudaGetLastError());
	CK(cudaMemcpyAsync(m->h_route_flag.get(), &M.route->overflow, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
	CK(cudaMemcpyAsync(m->h_ctr.get(), M.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
	p.valid = true;
	m->route_stage = 1;
	if (copied) CK(cudaEventSynchronize(m->ev_copied));
	return UFO_B200_OK;
}

int do_route_apply(Map* m, uint32_t first, uint32_t count, int last)
{
	if (!m) return UFO_B200_E_INVALID;
	DeviceMap& M = m->M;
	if (m->route_stage != 1 || first + count > M.route_world) {
		m->set_error("ufo_b200_route_apply without a marked pass, or sources out of range");
		return UFO_B200_E_INVALID;
	}
	CK(cudaSetDevice(m->device));
	cudaStream_t s = m->stream;
	PendingScan& p = m->pending;
	// every apply call is a scan of its own as far as the touched list goes: the first one starts
	// from the own bricks that kept local marks (list built by k_outbox under scan id + 1), the
	// following ones from an empty list
	M.scan_id += 1;
	if (M.scan_id == 0) M.scan_id = 1;
	if (!p.a.seg_cap) {  // first apply call of this pass (seg_cap is unused in routed passes: reused as a flag)
		std::swap(M.touched, M.touched_alt);
		std::swap(M.touched_mi, M.touched_alt_mi);
		M.dense = 0;
		M.mask_base = M.miss_mask;
		M.up_epoch++;
		if (M.up_epoch == 0) M.up_epoch = 1;
		p.a.seg_cap = 1;
	} else {
		CK(cudaMemsetAsync(&M.ctr->n_touched, 0, sizeof(uint32_t), s));
	}
	k_inbox<<<m->sm_count * 4, 256, 0, s>>>(M, first, count);
	++m->launches;
	launch_update(m, p.a.miss, false);
	launch_upper_seed(m);
	if (last) {
		if (m->profiling) CK(cudaEventRecord(m->ev[5], s));
		launch_upper_levels(m);
		CK(cudaEventRecord(m->ev[6], s));
		m->ev_valid = true;
		CK(cudaMemcpyAsync(m->h_ctr.get(), M.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
		m->stats_pending = true;
		m->route_stage = 2;
	}
	CK(cudaGetLastError());
	return UFO_B200_OK;
}

template <class F>
int guarded(Map* m, F&& f)
{
	if (m && m->device == -2) {
		m->set_error("geometry-only handle: no CUDA device bound");
		return UFO_B200_E_CUDA;
	}
	try {
		return f();
	} catch (CudaError& e) {
		if (m) m->set_error("CUDA error %s (%d) at ufo_map.cu:%d: %s", cudaGetErrorName(e.e), (int)e.e, e.line, e.what);
		return UFO_B200_E_CUDA;
	} catch (MapError& e) {
		return e.code;
	} catch (std::bad_alloc&) {
		if (m) m->set_error("out of memory");
		return UFO_B200_E_NOMEM;
	}
}

// Copies the first k entries of a device result list back to the caller's arrays (null ones are
// skipped); colours are packed r | g << 8 | b << 16 on the device, 3 bytes on the host.  Waits for s.
void copy_results(cudaStream_t s, size_t k, const unsigned long long* d_codes, uint64_t* codes, const float* d_occ,
                  float* logodds, const uint32_t* d_rgb, uint8_t* rgb)
{
	if (codes) CK(cudaMemcpyAsync(codes, d_codes, k * 8, cudaMemcpyDeviceToHost, s));
	if (logodds) CK(cudaMemcpyAsync(logodds, d_occ, k * 4, cudaMemcpyDeviceToHost, s));
	std::vector<uint32_t> h(rgb ? k : 0);
	if (rgb) CK(cudaMemcpyAsync(h.data(), d_rgb, k * 4, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	for (size_t i = 0; i < h.size(); ++i) {
		rgb[3 * i] = h[i] & 0xff;
		rgb[3 * i + 1] = (h[i] >> 8) & 0xff;
		rgb[3 * i + 2] = (h[i] >> 16) & 0xff;
	}
}

// launch(codes, occ, rgb, cap, count) enqueues kernels that count results into count and write the
// first cap of them to the lists (cap is 0 while the caller asks for the count only).  *n = the
// count; what fits in the caller's arrays is copied back.
template <class Launch>
void collect_results(Map* m, uint64_t* codes, float* logodds, uint8_t* rgb, size_t cap, size_t* n, Launch&& launch)
{
	cudaStream_t s = m->stream;
	const bool fill = codes != nullptr && cap > 0;
	Buffer<unsigned long long> d_count, d_codes;
	Buffer<float> d_occ;
	Buffer<uint32_t> d_rgb;
	d_count.resize(1, 0, s);
	if (fill) {
		d_codes.resize(cap);
		d_occ.resize(cap);
		if (rgb) d_rgb.resize(cap);
	}
	launch(d_codes.get(), d_occ.get(), d_rgb.get(), fill ? cap : 0, d_count.get());
	CK(cudaGetLastError());
	unsigned long long cnt = 0;
	CK(cudaMemcpyAsync(&cnt, d_count.get(), 8, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	*n = (size_t)cnt;
	if (fill) copy_results(s, std::min<size_t>(cnt, cap), d_codes.get(), codes, d_occ.get(), logodds, d_rgb.get(), rgb);
}
}  // namespace

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
extern "C" {

const char* ufo_b200_version(void) { return "ufomap_b200 0.1 (sm_100a)"; }

void ufo_b200_default_params(ufo_b200_params* p)
{
	if (!p) return;
	memset(p, 0, sizeof(*p));
	p->resolution = 0.1;
	p->depth_levels = 16;
	p->automatic_pruning = 1;
	p->occupied_thres = 0.5;
	p->free_thres = 0.5;
	p->prob_hit = 0.7;
	p->prob_miss = 0.4;
	p->clamping_thres_min = 0.1192;
	p->clamping_thres_max = 0.971;
	p->color = 0;
	p->device = -1;
}

int ufo_b200_create(const ufo_b200_params* p, ufo_b200_map** out)
{
	if (!p || !out) return UFO_B200_E_INVALID;
	*out = nullptr;
	if (p->depth_levels < 2 || p->depth_levels > 21 || !(p->resolution > 0)) return UFO_B200_E_INVALID;
	Map* m = new (std::nothrow) Map;
	if (!m) return UFO_B200_E_NOMEM;
	if (p->device == -2) {
		// geometry-only handle: indexing / computeRay helpers run on the host and need no
		// device; every call that touches map state fails with UFO_B200_E_CUDA
		m->device = -2;
		m->params = *p;
		m->M.g = make_geometry(p->resolution, p->depth_levels);
		m->occ_thr_log = to_logit(p->occupied_thres);
		m->free_thr_log = to_logit(p->free_thres);
		m->hit_log = to_logit(p->prob_hit);
		m->miss_log = to_logit(p->prob_miss);
		m->cmin_log = to_logit(p->clamping_thres_min);
		m->cmax_log = to_logit(p->clamping_thres_max);
		*out = m;
		return UFO_B200_OK;
	}
	int rc = guarded(m, [&]() {
		int dev = p->device;
		if (dev < 0) CK(cudaGetDevice(&dev));
		CK(cudaSetDevice(dev));
		m->device = dev;
		cudaDeviceProp prop;
		CK(cudaGetDeviceProperties(&prop, dev));
		m->sm_count = prop.multiProcessorCount;
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&m->ray_blocks_per_sm, k_rays<0, false>, kRayThreads, 0));
		if (m->ray_blocks_per_sm < 1) m->ray_blocks_per_sm = 1;
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&m->walk_blocks_per_sm, k_walk_mark<0, false, false, true>, kWalkThreads, 0));
		if (m->walk_blocks_per_sm < 1) m->walk_blocks_per_sm = 1;
		{
			const char* e = getenv("UFO_B200_MARK");
			m->force_records = e && !strcmp(e, "records");
			m->no_dense = e && !strcmp(e, "probe");
			// resident CTAs per SM of the two long kernels (tuning / co-residency experiments)
			const char* kb = getenv("UFO_B200_K3_BLOCKS");
			if (kb && atoi(kb) > 0) m->k3_blocks = atoi(kb);
			const char* wb = getenv("UFO_B200_WALK_BLOCKS");
			if (wb && atoi(wb) > 0) m->walk_blocks_per_sm = std::min(m->walk_blocks_per_sm, atoi(wb));
		}
		m->params = *p;
		CK(cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking));
		CK(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
		CK(cudaEventCreate(&m->ev_copy0));
		CK(cudaEventCreate(&m->ev_copied));
		m->stream = m->own_stream;
		for (auto& e : m->ev) CK(cudaEventCreate(&e));
		m->h_ctr.resize(1);
		m->M.g = make_geometry(p->resolution, p->depth_levels);
		m->M.color = p->color ? 1u : 0u;
		m->M.shard_rank = 0;
		m->M.shard_world = 1;
		m->occ_thr_log = to_logit(p->occupied_thres);
		m->free_thr_log = to_logit(p->free_thres);
		m->hit_log = to_logit(p->prob_hit);
		m->miss_log = to_logit(p->prob_miss);
		m->cmin_log = to_logit(p->clamping_thres_min);
		m->cmax_log = to_logit(p->clamping_thres_max);
		refresh_model(m);
		// a brick owns 64 block slots; the block hint is honoured through its brick equivalent
		// (a touched brick of a lidar scan holds ~32 touched blocks)
		uint64_t bricks64 = p->initial_bricks ? p->initial_bricks
		                                      : (p->initial_blocks ? p->initial_blocks / 32 : (1ull << 15));
		uint32_t bricks = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(bricks64, 16), 0x3ffffffull);
		uint32_t upper = std::max(bricks / 2, 4096u);
		alloc_pools(m, bricks, upper);
		m->n_blocks = 0;
		m->n_bricks = 0;
		m->n_upper = 0;
		reset_bbox(m);
		CK(cudaStreamSynchronize(m->stream));
		return (int)UFO_B200_OK;
	});
	if (rc != UFO_B200_OK) {
		fprintf(stderr, "ufo_b200_create failed: %s\n", m->err.c_str());
		ufo_b200_destroy(m);
		return rc;
	}
	*out = m;
	return UFO_B200_OK;
}

void ufo_b200_destroy(ufo_b200_map* m)
{
	if (!m) return;
	if (m->device != -2) {
		cudaSetDevice(m->device);
		cudaStreamSynchronize(m->stream);
	}
	delete m;
}

const char* ufo_b200_last_error(const ufo_b200_map* m) { return m ? m->err.c_str() : "null map"; }

int ufo_b200_set_stream(ufo_b200_map* m, void* cuda_stream)
{
	if (!m) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		sync_map(m);
		m->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : m->own_stream;
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_insert_pointcloud(ufo_b200_map* m, const double origin[3], const void* points,
                               size_t n, int layout, double max_range, uint32_t depth,
                               int simple_ray_casting, uint32_t early_stopping, int discrete,
                               int async)
{
	return guarded(m, [&]() {
		return do_insert(m, origin, points, false, n, nullptr, layout, max_range, depth,
		                 simple_ray_casting, early_stopping, discrete, async);
	});
}

int ufo_b200_insert_device(ufo_b200_map* m, const double origin[3], const void* d_points,
                           size_t n, int layout, double max_range, uint32_t depth,
                           int simple_ray_casting, uint32_t early_stopping, int discrete,
                           int async)
{
	return guarded(m, [&]() {
		return do_insert(m, origin, d_points, true, n, nullptr, layout, max_range, depth,
		                 simple_ray_casting, early_stopping, discrete, async);
	});
}

int ufo_b200_insert_pointcloud_frame(ufo_b200_map* m, const double origin[3], const void* points,
                                     size_t n, int layout, const double frame_pose[7],
                                     double max_range, uint32_t depth, int simple_ray_casting,
                                     uint32_t early_stopping, int discrete, int async)
{
	if (m && !frame_pose) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		return do_insert(m, origin, points, false, n, frame_pose, layout, max_range, depth,
		                 simple_ray_casting, early_stopping, discrete, async);
	});
}

int ufo_b200_insert_pointcloud2(ufo_b200_map* m, const double origin[3], const ufo_b200_cloud2* cloud,
                                const double* frame_pose, double max_range, uint32_t depth,
                                int simple_ray_casting, uint32_t early_stopping, int discrete, int async)
{
	if (m && !cloud) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		return do_insert(m, origin, cloud->data, cloud->on_device != 0, cloud->n, frame_pose, 4, max_range,
		                 depth, simple_ray_casting, early_stopping, discrete, async, cloud);
	});
}

int ufo_b200_transform_points(const double frame_pose[7], const void* points, size_t n, int layout,
                              double* out_xyz)
{
	if (!frame_pose || (n && (!points || !out_xyz)) || layout < 0 || layout > 3)
		return UFO_B200_E_INVALID;
	const Frame f{frame_pose[3], frame_pose[4], frame_pose[5], frame_pose[6],
	              frame_pose[0], frame_pose[1], frame_pose[2]};
	const size_t stride = (layout == UFO_B200_XYZ_F64 || layout == UFO_B200_XYZ_F32) ? 3 : 4;
	const bool f64 = layout == UFO_B200_XYZ_F64 || layout == UFO_B200_XYZRGB_F64;
	for (size_t i = 0; i < n; ++i) {
		Vec3 p;
		if (f64) {
			const double* q = static_cast<const double*>(points) + stride * i;
			p = {q[0], q[1], q[2]};
		} else {
			const float* q = static_cast<const float*>(points) + stride * i;
			p = {(double)q[0], (double)q[1], (double)q[2]};
		}
		Vec3 r = frame_transform(f, p);
		out_xyz[3 * i + 0] = r.x;
		out_xyz[3 * i + 1] = r.y;
		out_xyz[3 * i + 2] = r.z;
	}
	return UFO_B200_OK;
}

int ufo_b200_pose_from_rpy(double x, double y, double z, double roll, double pitch, double yaw,
                           double frame_pose[7])
{
	if (!frame_pose) return UFO_B200_E_INVALID;
	// Quaternion(roll, pitch, yaw) of the reference goes through the ZYX rotation matrix and the
	// trace formulas (math/quaternion.h:69-93); restated with the same expression order.
	const double sr = sin(roll), sp = sin(pitch), sy = sin(yaw);
	const double cr = cos(roll), cp = cos(pitch), cy = cos(yaw);
	const double m00 = cy * cp, m01 = cy * sp * sr - sy * cr, m02 = cy * sp * cr + sy * sr;
	const double m10 = sy * cp, m11 = sy * sp * sr + cy * cr, m12 = sy * sp * cr - cy * sr;
	const double m20 = -sp, m21 = cp * sr, m22 = cp * cr;
	const double qw = sqrt(std::max(0.0, 1 + m00 + m11 + m22)) / 2.0;
	const double ax = sqrt(std::max(0.0, 1 + m00 - m11 - m22)) / 2.0;
	const double ay = sqrt(std::max(0.0, 1 - m00 + m11 - m22)) / 2.0;
	const double az = sqrt(std::max(0.0, 1 - m00 - m11 + m22)) / 2.0;
	frame_pose[0] = x;
	frame_pose[1] = y;
	frame_pose[2] = z;
	frame_pose[3] = qw;
	frame_pose[4] = (m21 - m12) >= 0 ? fabs(ax) : -fabs(ax);
	frame_pose[5] = (m02 - m20) >= 0 ? fabs(ay) : -fabs(ay);
	frame_pose[6] = (m10 - m01) >= 0 ? fabs(az) : -fabs(az);
	return UFO_B200_OK;
}

int ufo_b200_wait(ufo_b200_map* m)
{
	if (!m) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		return sync_map(m);
	});
}

int ufo_b200_done(ufo_b200_map* m, int* done)
{
	if (!m || !done) return UFO_B200_E_INVALID;
	if (m->device == -2) return UFO_B200_E_CUDA;
	cudaError_t e = cudaStreamQuery(m->stream);
	if (e == cudaSuccess) {
		// the stream is idle; if the scan ran into a full pool it is not integrated yet: grow and repeat
		// it now, so that a caller polling this function always gets to "done"
		if (m->pending.valid && m->h_ctr->overflow) {
			const int rc = guarded(m, [&]() {
				CK(cudaSetDevice(m->device));
				return sync_map(m);
			});
			if (rc != UFO_B200_OK) return rc;
		}
		*done = 1;
		return UFO_B200_OK;
	}
	if (e == cudaErrorNotReady) {
		*done = 0;
		return UFO_B200_OK;
	}
	m->set_error("cudaStreamQuery: %s", cudaGetErrorString(e));
	return UFO_B200_E_CUDA;
}

int ufo_b200_compute_ray(const ufo_b200_map* m, const double origin[3], const double end_in[3],
                         double max_range, uint32_t depth, uint64_t* codes, size_t cap, size_t* n)
{
	if (!m || !origin || !end_in || !n) return UFO_B200_E_INVALID;
	const Geometry& g = m->M.g;
	Vec3 o = {origin[0], origin[1], origin[2]}, e = {end_in[0], end_in[1], end_in[2]};
	Vec3 dir = vsub(e, o);
	double dist = vnorm(dir);
	dir = vdiv(dir, dist);
	if (0 <= max_range && dist > max_range) {
		e = vadd(o, vscale(dir, max_range));
		dist = max_range;
	}
	Walk w;
	walk_init(g, o, e, dir, depth, w);
	size_t cnt = 0;
	if (!w.same) {
		while (w.cur != w.end && walk_tmin(w) <= dist) {
			if (codes && cnt < cap) codes[cnt] = key_to_code(w.cur);
			++cnt;
			walk_step(w);
		}
	}
	*n = cnt;
	return UFO_B200_OK;
}

int ufo_b200_to_key(const ufo_b200_map* m, const double xyz[3], uint32_t depth, uint32_t key[3])
{
	if (!m || !xyz || !key) return UFO_B200_E_INVALID;
	Key3 k = point_to_key(m->M.g, {xyz[0], xyz[1], xyz[2]}, depth);
	key[0] = k.x;
	key[1] = k.y;
	key[2] = k.z;
	return UFO_B200_OK;
}

int ufo_b200_to_code(const ufo_b200_map* m, const double xyz[3], uint32_t depth, uint64_t* code)
{
	if (!m || !xyz || !code) return UFO_B200_E_INVALID;
	*code = key_to_code(point_to_key(m->M.g, {xyz[0], xyz[1], xyz[2]}, depth));
	return UFO_B200_OK;
}

int ufo_b200_key_to_coord(const ufo_b200_map* m, const uint32_t key[3], uint32_t depth, double xyz[3])
{
	if (!m || !key || !xyz) return UFO_B200_E_INVALID;
	Vec3 p = key_to_coord(m->M.g, {key[0], key[1], key[2]}, depth);
	xyz[0] = p.x;
	xyz[1] = p.y;
	xyz[2] = p.z;
	return UFO_B200_OK;
}

uint64_t ufo_b200_key_to_code(const uint32_t key[3]) { return key_to_code({key[0], key[1], key[2]}); }

void ufo_b200_code_to_key(uint64_t code, uint32_t key[3])
{
	Key3 k = code_to_key(code);
	key[0] = k.x;
	key[1] = k.y;
	key[2] = k.z;
}

int ufo_b200_query(ufo_b200_map* m, const uint64_t* codes, const uint32_t* depths, size_t n,
                   float* logodds, uint8_t* flags, uint8_t* rgb)
{
	if (!m || (n && (!codes || !depths || !logodds || !flags))) return UFO_B200_E_INVALID;
	if (!n) return UFO_B200_OK;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		sync_map(m);
		cudaStream_t s = m->stream;
		Buffer<unsigned long long> d_codes;
		Buffer<uint32_t> d_depths, d_rgb;
		Buffer<float> d_occ;
		Buffer<uint8_t> d_flags;
		d_codes.resize(n);
		d_depths.resize(n);
		d_occ.resize(n);
		d_flags.resize(n);
		if (rgb) d_rgb.resize(n);
		CK(cudaMemcpyAsync(d_codes.get(), codes, n * 8, cudaMemcpyHostToDevice, s));
		CK(cudaMemcpyAsync(d_depths.get(), depths, n * 4, cudaMemcpyHostToDevice, s));
		k_query<<<(uint32_t)((n + 255) / 256), 256, 0, s>>>(m->M, d_codes.get(), d_depths.get(), (uint32_t)n, d_occ.get(),
		                                                    d_flags.get(), d_rgb.get());
		CK(cudaGetLastError());
		CK(cudaMemcpyAsync(flags, d_flags.get(), n, cudaMemcpyDeviceToHost, s));
		copy_results(s, n, nullptr, nullptr, d_occ.get(), logodds, d_rgb.get(), rgb);
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_export_leaves(ufo_b200_map* m, uint64_t* codes, float* logodds, uint8_t* rgb,
                           size_t cap, size_t* n)
{
	if (!m || !n) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		sync_map(m);
		collect_results(m, codes, logodds, rgb, cap, n, [&](unsigned long long* d_codes, float* d_occ, uint32_t* d_rgb,
		                                                     size_t d_cap, unsigned long long* d_count) {
			const size_t threads = (size_t)m->n_bricks * 64 * 64;
			if (threads)
				k_export<<<(uint32_t)((threads + 255) / 256), 256, 0, m->stream>>>(m->M, m->n_bricks, d_codes, d_occ, d_rgb, d_cap, d_count);
		});
		return (int)UFO_B200_OK;
	});
}

}  // extern "C"

namespace
{
// ---- file image (ufo_export.cuh): the levels above the bricks, on the host ----
struct UpNode {
	int32_t child[8];  // -1: absent; >= 0: index into nodes (depth > 5) or into the sorted brick list (depth 5)
	uint8_t mask;      // children written as records (they have children and lie above min_depth)
	uint8_t hit;       // children whose cube intersects the export box
	bool has;          // false: collapsed to a leaf (canonical export only)
	float occ;
	uint32_t rgb;
	unsigned long long size;  // bytes of the node's record
};

struct ExportPlan {
	std::vector<uint32_t> order;  // bricks of the map in Morton (= stream) order
	std::vector<BrickInfo> info;  // indexed by brick slot
	std::vector<UpNode> nodes;    // nodes[0] = root (if any brick exists)
	std::vector<unsigned long long> codes;
	uint32_t P = 4;
	uint32_t levels = 16;
	uint32_t min_depth = 0;
	bool pruned = false;
	ExportBox box{};
	const Geometry* g = nullptr;
};

unsigned long long spread3_host(unsigned long long v)
{
	unsigned long long r = 0;
	for (int i = 0; i < 21; ++i) r |= ((v >> i) & 1ull) << (3 * i);
	return r;
}

// builds the node of depth d (centre c) that covers order[lo, hi); returns its index in plan.nodes
int32_t build_upper(ExportPlan& plan, uint32_t d, size_t lo, size_t hi, const double c[3])
{
	const int32_t self = (int32_t)plan.nodes.size();
	plan.nodes.push_back(UpNode{});
	UpNode n{};
	n.has = true;
	n.size = 1;
	const uint32_t shift = 3 * (d - 5);  // child index of a depth-d node inside the brick code
	const double chs = plan.g->half_size[d - 1];
	float occ[8];
	uint32_t rgb[8];
	bool any_children = false;
	size_t pos = lo;
	for (uint32_t i = 0; i < 8; ++i) {
		size_t end = pos;
		while (end < hi && ((plan.codes[end] >> shift) & 7ull) == i) ++end;
		double cc[3];
		child_center(c, chs, i, cc);
		const bool hit = box_hits(plan.box, cc, chs);
		if (hit) n.hit |= (uint8_t)(1u << i);
		n.child[i] = -1;
		occ[i] = 0.0f;
		rgb[i] = 0;
		unsigned long long bytes = plan.P;  // absent child: one default payload
		if (end > pos) {
			if (d == 5) {
				const BrickInfo& bi = plan.info[plan.order[pos]];
				n.child[i] = (int32_t)pos;
				occ[i] = bi.occ;
				rgb[i] = bi.rgb;
				if (bi.flags & 1u) {
					any_children = true;
					if (plan.min_depth < 4) n.mask |= (uint8_t)(1u << i);
				}
				bytes = bi.size;  // 0 when the brick's cube misses the box (same test on the device)
			} else {
				const int32_t ci = build_upper(plan, d - 1, pos, end, cc);
				const UpNode& ch = plan.nodes[ci];
				n.child[i] = ci;
				occ[i] = ch.occ;
				rgb[i] = ch.rgb;
				if (ch.has) {
					any_children = true;
					n.mask |= (uint8_t)(1u << i);  // d - 1 >= 5 > min_depth
					bytes = ch.size;
				}
			}
		}
		if (hit) n.size += bytes;
		pos = end;
	}
	if (plan.pruned && !any_children) {
		bool same = true;
		for (int i = 1; i < 8; ++i) same = same && occ[i] == occ[0] && rgb[i] == rgb[0];
		if (same) n.has = false;
	}
	n.occ = occ[0];  // payload if collapsed
	n.rgb = rgb[0];
	plan.nodes[self] = n;
	return self;
}

template <class Sink>
void put_payload_host(Sink& sink, uint32_t P, float occ, uint32_t rgb)
{
	uint8_t b[7];
	std::memcpy(b, &occ, 4);
	b[4] = (uint8_t)rgb;
	b[5] = (uint8_t)(rgb >> 8);
	b[6] = (uint8_t)(rgb >> 16);
	sink(b, P);
}

template <class Sink>
void emit_upper(const ExportPlan& plan, const std::vector<unsigned long long>& offs, const uint8_t* packed,
                int32_t idx, uint32_t d, Sink& sink)
{
	const UpNode& n = plan.nodes[idx];
	sink(&n.mask, 1);
	for (uint32_t i = 0; i < 8; ++i) {
		if (!((n.hit >> i) & 1u)) continue;
		const int32_t c = n.child[i];
		if (c < 0) {
			put_payload_host(sink, plan.P, 0.0f, 0u);
		} else if (d == 5) {
			const uint32_t slot = plan.order[c];
			const BrickInfo& bi = plan.info[slot];
			if (bi.size == 0) continue;
			if (bi.flags & 4u) sink(packed + offs[slot], bi.size);
			else put_payload_host(sink, plan.P, bi.occ, bi.rgb);
		} else if (plan.nodes[c].has) {
			emit_upper(plan, offs, packed, c, d - 1, sink);
		} else {
			put_payload_host(sink, plan.P, plan.nodes[c].occ, plan.nodes[c].rgb);
		}
	}
}

// Produces the node stream (optionally behind the file header) through sink(ptr, len) calls, in
// order.  *total = bytes produced.
template <class Sink>
int export_image(Map* m, int pruned, uint32_t min_depth, const double* box6, bool with_header, Sink&& sink,
                 unsigned long long* total)
{
	if (m->device == -2) return UFO_B200_E_CUDA;
	if (m->M.g.depth_levels < 5) {
		m->set_error("export needs depth_levels >= 5");
		return UFO_B200_E_UNSUPPORTED;
	}
	if (min_depth > 4) {
		m->set_error("export with min_depth %u > 4 is not supported", min_depth);
		return UFO_B200_E_UNSUPPORTED;
	}
	CK(cudaSetDevice(m->device));
	sync_map(m);
	cudaStream_t s = m->stream;
	const uint32_t nb = m->n_bricks;
	const bool color = m->M.color != 0;
	ExportPlan plan;
	plan.P = color ? 7 : 4;
	plan.levels = m->M.g.depth_levels;
	plan.min_depth = min_depth;
	plan.pruned = pruned != 0;
	plan.g = &m->M.g;
	if (box6) {
		// the reference's AABB stores centre and half size (geometry/aabb.h:49-70); getMin/getMax
		plan.box.on = 1;
		for (int k = 0; k < 3; ++k) {
			plan.box.lo[k] = box6[k] - box6[3 + k];
			plan.box.hi[k] = box6[k] + box6[3 + k];
		}
	}
	*total = 0;
	const double c0[3] = {0.0, 0.0, 0.0};
	auto header = [&](char* head, size_t cap, unsigned long long data_size) {
		// octree.h:850-860; doubles print with the default ostream precision = %g
		return snprintf(head, cap,
		                "# UFOMap file\n# (feel free to add / change comments, but leave the first line as it "
		                "is!)\n#\nversion 1.0.0\nid %s\nresolution %g\ndepth_levels %u\ncompressed 0\n"
		                "uncompressed_data_size %d\ndata\n",
		                color ? "occupancy_map_color" : "occupancy_map", m->M.g.resolution, plan.levels, (int)data_size);
	};
	if (!box_hits(plan.box, c0, plan.g->half_size[plan.levels])) {
		// "No node intersects": the reference writes no node data at all (OMB:1462-1468)
		if (with_header) {
			char head[512];
			const int hl = header(head, sizeof head, 0);
			sink(head, (size_t)hl);
			*total = (unsigned long long)hl;
		}
		return UFO_B200_OK;
	}
	plan.info.resize(nb);
	std::vector<unsigned long long> keys(nb);
	Buffer<BrickInfo> d_info;
	Buffer<unsigned long long> d_offs;
	Buffer<uint8_t> d_out;
	if (nb) {
		d_info.resize(nb);
		if (color) k_brick_stream<true><<<nb, 64, 0, s>>>(m->M, nb, pruned, min_depth, plan.box, d_info.get(), nullptr, nullptr);
		else k_brick_stream<false><<<nb, 64, 0, s>>>(m->M, nb, pruned, min_depth, plan.box, d_info.get(), nullptr, nullptr);
		CK(cudaGetLastError());
		CK(cudaMemcpyAsync(plan.info.data(), d_info.get(), sizeof(BrickInfo) * nb, cudaMemcpyDeviceToHost, s));
		CK(cudaMemcpyAsync(keys.data(), m->M.brick_key, 8ull * nb, cudaMemcpyDeviceToHost, s));
		CK(cudaStreamSynchronize(s));
	}
	// bricks that are part of the tree, in Morton order; a leaf brick with the default payload is
	// indistinguishable from untouched space
	std::vector<std::pair<unsigned long long, uint32_t>> sorted;
	sorted.reserve(nb);
	for (uint32_t b = 0; b < nb; ++b) {
		const BrickInfo& bi = plan.info[b];
		if (bi.flags & 2u) continue;
		if (!(bi.flags & 1u) && bi.occ == 0.0f && bi.rgb == 0u) continue;
		uint32_t x, y, z;
		unpack_key(keys[b], x, y, z);
		sorted.emplace_back(spread3_host(x) | (spread3_host(y) << 1) | (spread3_host(z) << 2), b);
	}
	std::sort(sorted.begin(), sorted.end());
	plan.order.resize(sorted.size());
	plan.codes.resize(sorted.size());
	std::vector<unsigned long long> offs(nb, ~0ull);
	unsigned long long packed_bytes = 0;
	for (size_t i = 0; i < sorted.size(); ++i) {
		plan.codes[i] = sorted[i].first;
		plan.order[i] = sorted[i].second;
		const BrickInfo& bi = plan.info[sorted[i].second];
		if (bi.flags & 4u) {
			offs[sorted[i].second] = packed_bytes;
			packed_bytes += bi.size;
		}
	}
	bool root_has = false;
	unsigned long long data_size = 1 + plan.P;  // children byte + root payload
	if (!sorted.empty()) {
		build_upper(plan, plan.levels, 0, sorted.size(), c0);
		root_has = plan.nodes[0].has;
		if (root_has) data_size = 1 + plan.nodes[0].size;
	}
	std::vector<uint8_t> packed(packed_bytes);
	if (packed_bytes) {
		d_offs.resize(nb);
		d_out.resize(packed_bytes);
		CK(cudaMemcpyAsync(d_offs.get(), offs.data(), 8ull * nb, cudaMemcpyHostToDevice, s));
		if (color) k_brick_stream<true><<<nb, 64, kBrickStreamMax, s>>>(m->M, nb, pruned, min_depth, plan.box, d_info.get(), d_offs.get(), d_out.get());
		else k_brick_stream<false><<<nb, 64, kBrickStreamMax, s>>>(m->M, nb, pruned, min_depth, plan.box, d_info.get(), d_offs.get(), d_out.get());
		CK(cudaGetLastError());
		CK(cudaMemcpyAsync(packed.data(), d_out.get(), packed_bytes, cudaMemcpyDeviceToHost, s));
		CK(cudaStreamSynchronize(s));
	}
	unsigned long long produced = 0;
	auto counted = [&](const void* p, size_t len) {
		sink(p, len);
		produced += len;
	};
	if (with_header) {
		char head[512];
		const int hl = header(head, sizeof head, data_size);
		counted(head, (size_t)hl);
	}
	const uint8_t children = root_has ? 0xff : 0x00;
	counted(&children, 1);
	if (root_has) {
		emit_upper(plan, offs, packed.data(), 0, plan.levels, counted);
	} else {
		const float occ = sorted.empty() ? 0.0f : plan.nodes[0].occ;
		const uint32_t rgb = sorted.empty() ? 0u : plan.nodes[0].rgb;
		put_payload_host(counted, plan.P, occ, rgb);
	}
	*total = produced;
	return UFO_B200_OK;
}
}  // namespace

namespace
{
// LZ4 block API of the system's liblz4 (the reference links it: octree.h:1428-1486), loaded on
// first use so that the library does not depend on LZ4 development files.
struct Lz4 {
	int (*bound)(int) = nullptr;
	int (*fast)(const char*, char*, int, int, int) = nullptr;
	int (*hc)(const char*, char*, int, int, int) = nullptr;
	int (*decompress)(const char*, char*, int, int) = nullptr;
	bool ok = false;
};

const Lz4& lz4()
{
	static Lz4 api = []() {
		Lz4 a;
		void* h = dlopen("liblz4.so.1", RTLD_NOW | RTLD_LOCAL);
		if (!h) h = dlopen("liblz4.so", RTLD_NOW | RTLD_LOCAL);
		if (h) {
			a.bound = reinterpret_cast<int (*)(int)>(dlsym(h, "LZ4_compressBound"));
			a.fast = reinterpret_cast<int (*)(const char*, char*, int, int, int)>(dlsym(h, "LZ4_compress_fast"));
			a.hc = reinterpret_cast<int (*)(const char*, char*, int, int, int)>(dlsym(h, "LZ4_compress_HC"));
			a.decompress = reinterpret_cast<int (*)(const char*, char*, int, int)>(dlsym(h, "LZ4_decompress_safe"));
			a.ok = a.bound && a.fast && a.hc && a.decompress;
		}
		return a;
	}();
	return api;
}

// compressData (octree.h:1428-1456): the whole node stream as ONE LZ4 block
bool lz4_compress(const std::vector<uint8_t>& in, int acceleration, int level, std::vector<uint8_t>& out)
{
	const Lz4& z = lz4();
	if (!z.ok || in.size() > 0x7e000000u) return false;
	const int cap = z.bound((int)in.size());
	out.resize((size_t)std::max(cap, 1));
	const int n = level <= 0 ? z.fast(reinterpret_cast<const char*>(in.data()), reinterpret_cast<char*>(out.data()), (int)in.size(), cap, acceleration)
	                         : z.hc(reinterpret_cast<const char*>(in.data()), reinterpret_cast<char*>(out.data()), (int)in.size(), cap, level);
	if (n < 0) return false;
	out.resize((size_t)n);
	return true;
}
}  // namespace

extern "C" {

int ufo_b200_set_value_volume(ufo_b200_map* m, const double box6[6], double occupancy, uint32_t min_depth)
{
	if (!m || !box6) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		if (min_depth > 4 || m->M.g.depth_levels < 5) {
			m->set_error("setValueVolume: min_depth %u > 4 (or depth_levels < 5) is not supported", min_depth);
			return (int)UFO_B200_E_UNSUPPORTED;
		}
		if (m->M.color && min_depth > 0) {
			m->set_error("setValueVolume on a colour map is supported at min_depth 0 only");
			return (int)UFO_B200_E_UNSUPPORTED;
		}
		if (m->M.shard_world > 1) {
			m->set_error("setValueVolume on a sharded map is not supported");
			return (int)UFO_B200_E_UNSUPPORTED;
		}
		const Geometry& g = m->M.g;
		VolumeArgs v{};
		v.min_depth = min_depth;
		v.box.on = 1;
		for (int k = 0; k < 3; ++k) {
			v.box.lo[k] = box6[k] - box6[3 + k];
			v.box.hi[k] = box6[k] + box6[3 + k];
		}
		const double c0[3] = {0.0, 0.0, 0.0};
		if (!box_hits(v.box, c0, g.half_size[g.depth_levels])) return (int)UFO_B200_OK;  // no node intersects
		// candidate bricks: the key range of the box, one brick of slack on every side (the kernel
		// decides with the reference's own cube tests)
		const double ext = g.half_size[g.depth_levels];
		const long long top = (1ll << (g.depth_levels - 4)) - 1;
		uint32_t first[3], count[3];
		unsigned long long total = 1;
		for (int k = 0; k < 3; ++k) {
			const double lo = std::max(v.box.lo[k], -ext), hi = std::min(v.box.hi[k], ext);
			long long a = ((long long)std::floor(lo * g.resolution_factor) + (long long)g.max_value) >> 4;
			long long b = ((long long)std::floor(hi * g.resolution_factor) + (long long)g.max_value) >> 4;
			a = std::min(std::max(a - 1, 0ll), top);
			b = std::min(std::max(b + 1, 0ll), top);
			first[k] = (uint32_t)a;
			count[k] = (uint32_t)(b - a + 1);
			total *= count[k];
		}
		if (total > (1ull << 22)) {
			m->set_error("setValueVolume: the box covers %llu bricks (limit 4194304)", total);
			return (int)UFO_B200_E_UNSUPPORTED;
		}
		v.bx0 = first[0];
		v.by0 = first[1];
		v.bz0 = first[2];
		v.nx = count[0];
		v.ny = count[1];
		v.nz = count[2];
		// setOccupancy(LogitType&, LogitType const&): float clamp of the float logit (OMB:1151-1157)
		const float lo = (float)m->cmin_log, hi = (float)m->cmax_log;
		float value = (float)to_logit(occupancy);
		value = value < lo ? lo : (hi < value ? hi : value);
		const double origin[3] = {0.0, 0.0, 0.0};
		return do_insert(m, origin, nullptr, false, 0, nullptr, UFO_B200_XYZ_F64, -1.0, 0, 0, 0, 0, 0, nullptr, &v, value);
	});
}

int ufo_b200_write(ufo_b200_map* m, const double* box6, uint32_t min_depth, int expanded, void* buf, size_t cap,
                   size_t* size)
{
	if (!m || !size) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		uint8_t* out = static_cast<uint8_t*>(buf);
		size_t at = 0;
		unsigned long long total = 0;
		int rc = export_image(m, expanded ? 0 : 1, min_depth, box6, true, [&](const void* p, size_t len) {
			if (out && at + len <= cap) std::memcpy(out + at, p, len);
			at += len;
		}, &total);
		*size = (size_t)total;
		return rc;
	});
}

int ufo_b200_write_data(ufo_b200_map* m, const double* box6, uint32_t min_depth, void* buf, size_t cap,
                        size_t* size)
{
	if (!m || !size) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		uint8_t* out = static_cast<uint8_t*>(buf);
		size_t at = 0;
		unsigned long long total = 0;
		int rc = export_image(m, 1, min_depth, box6, false, [&](const void* p, size_t len) {
			if (out && at + len <= cap) std::memcpy(out + at, p, len);
			at += len;
		}, &total);
		*size = (size_t)total;
		return rc;
	});
}

int ufo_b200_write_file(ufo_b200_map* m, const char* filename, const double* box6, uint32_t min_depth,
                        int expanded)
{
	if (!m || !filename) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		FILE* f = fopen(filename, "wb");
		if (!f) {
			m->set_error("cannot open %s", filename);
			return (int)UFO_B200_E_INVALID;
		}
		unsigned long long total = 0;
		bool ok = true;
		int rc = export_image(m, expanded ? 0 : 1, min_depth, box6, true,
		                      [&](const void* p, size_t len) { ok = ok && fwrite(p, 1, len, f) == len; }, &total);
		ok = fclose(f) == 0 && ok;
		if (rc == UFO_B200_OK && !ok) {
			m->set_error("short write to %s", filename);
			return (int)UFO_B200_E_INVALID;
		}
		return rc;
	});
}

int ufo_b200_set_sensor_model(ufo_b200_map* m, const double p[6])
{
	if (!m || !p) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		sync_map(m);
		m->occ_thr_log = to_logit(p[0]);
		m->free_thr_log = to_logit(p[1]);
		m->hit_log = to_logit(p[2]);
		m->miss_log = to_logit(p[3]);
		m->cmin_log = to_logit(p[4]);
		m->cmax_log = to_logit(p[5]);
		refresh_model(m);
		rebuild_flags(m);
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_set_sensor_model_field(ufo_b200_map* m, int index, double probability)
{
	if (!m || index < 0 || index > 5) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		sync_map(m);
		double* field[6] = {&m->occ_thr_log, &m->free_thr_log, &m->hit_log, &m->miss_log, &m->cmin_log, &m->cmax_log};
		*field[index] = to_logit(probability);
		refresh_model(m);
		if (index <= 1) rebuild_flags(m);
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_sensor_model_logit(const ufo_b200_map* m, double o[6])
{
	if (!m || !o) return UFO_B200_E_INVALID;
	o[0] = m->occ_thr_log;
	o[1] = m->free_thr_log;
	o[2] = m->hit_log;
	o[3] = m->miss_log;
	o[4] = m->cmin_log;
	o[5] = m->cmax_log;
	return UFO_B200_OK;
}

int ufo_b200_change_bbox(ufo_b200_map* m, double mn[3], double mx[3])
{
	if (!m || !mn || !mx) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		sync_map(m);
		memcpy(mn, m->min_change, sizeof(m->min_change));
		memcpy(mx, m->max_change, sizeof(m->max_change));
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_reset_change_bbox(ufo_b200_map* m)
{
	if (!m) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		sync_map(m);
		reset_bbox(m);
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_last_scan_stats(ufo_b200_map* m, ufo_b200_scan_stats* out)
{
	if (!m || !out) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		sync_map(m);
		*out = m->stats;
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_completed_scan_stats(ufo_b200_map* m, ufo_b200_scan_stats* out)
{
	if (!m || !out) return UFO_B200_E_INVALID;
	*out = m->done_stats;
	return UFO_B200_OK;
}

int ufo_b200_set_profiling(ufo_b200_map* m, int enable)
{
	if (!m) return UFO_B200_E_INVALID;
	m->profiling = enable < 0 ? 0 : enable;
	return UFO_B200_OK;
}

int ufo_b200_set_shard(ufo_b200_map* m, uint32_t rank, uint32_t world)
{
	if (!m || (world > 1 && rank >= world)) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		sync_map(m);
		if (m->n_bricks != 0) {
			m->set_error("ufo_b200_set_shard must be called on an empty map");
			return (int)UFO_B200_E_INVALID;
		}
		m->M.shard_rank = world > 1 ? rank : 0;
		m->M.shard_world = world > 1 ? world : 1;
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_clear(ufo_b200_map* m)
{
	if (!m) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		try {
			sync_map(m);
		} catch (MapError&) {
			// a scan that failed half-way: its marks are wiped below
		}
		DeviceMap& M = m->M;
		cudaStream_t s = m->stream;
		m->bh_tab.fill(0xff, s);
		m->uh_keys.fill(0xff, s);
		m->uh_vals.fill(0xff, s);
		for_each_pool_array(m, [&](const PoolArray& a) {
			if (a.cleared && a.buf.get()) a.buf.fill(a.fill, s, in_use(m, a.unit) * a.unit_bytes);
		});
		if (m->vol.get()) wipe_volume(m);
		m->n_blocks = 0;
		m->n_bricks = 0;
		m->n_upper = 0;
		M.scan_id = 0;
		M.up_epoch = 0;
		m->poisoned = false;
		m->route_stage = 0;
		reset_bbox(m);
		CK(cudaStreamSynchronize(s));
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_clear_resize(ufo_b200_map* m, double resolution, uint32_t depth_levels)
{
	if (!m) return UFO_B200_E_INVALID;
	if (depth_levels < 2 || depth_levels > 21 || !(resolution > 0)) return UFO_B200_E_INVALID;  // octree.h:931-935
	int rc = ufo_b200_clear(m);
	if (rc != UFO_B200_OK) return rc;
	return guarded(m, [&]() {
		m->params.resolution = resolution;
		m->params.depth_levels = depth_levels;
		m->M.g = make_geometry(resolution, depth_levels);
		refresh_model(m);
		reset_bbox(m);
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_route_inbox_bytes(uint32_t world, uint32_t cap_bricks, uint32_t cap_hits, size_t* bytes)
{
	if (!bytes || world < 2 || world > kMaxRanks || !cap_bricks || !cap_hits) return UFO_B200_E_INVALID;
	*bytes = route_layout(world, cap_bricks, cap_hits, nullptr, nullptr, nullptr);
	return UFO_B200_OK;
}

int ufo_b200_route_setup(ufo_b200_map* m, uint32_t rank, uint32_t world, uint32_t cap_bricks, uint32_t cap_hits,
                         void** inbox)
{
	if (!m || !inbox || world < 2 || world > kMaxRanks || rank >= world || !cap_bricks || !cap_hits) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		sync_map(m);
		if (m->n_bricks != 0 || m->route_inbox.get() || m->M.shard_world > 1 || m->M.color) {
			m->set_error("ufo_b200_route_setup: needs an empty, unsharded mono map and may be called once");
			return (int)UFO_B200_E_INVALID;
		}
		const size_t total = route_layout(world, cap_bricks, cap_hits, &m->route_region, &m->route_miss_off, &m->route_hit_off);
		m->route_inbox.resize(total, 0);
		m->route.resize(1, 0);
		m->M.route = m->route.get();
		m->h_route.resize(1);
		m->h_route_flag.resize(1);
		*m->h_route_flag = 0;
		m->route_cap_m = cap_bricks;
		m->route_cap_h = cap_hits;
		m->M.route_rank = rank;
		m->M.route_world = world;
		*inbox = m->route_inbox.get();
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_route_connect(ufo_b200_map* m, void* const* peer_inboxes)
{
	if (!m || !peer_inboxes || m->M.route_world < 2) return UFO_B200_E_INVALID;
	for (uint32_t r = 0; r < m->M.route_world; ++r) {
		if (!peer_inboxes[r]) return UFO_B200_E_INVALID;
		m->route_peer[r] = peer_inboxes[r];
	}
	return UFO_B200_OK;
}

int ufo_b200_route_mark(ufo_b200_map* m, const double origin[3], const void* points, size_t n, int layout,
                        double max_range, int on_device, int self_too)
{
	return guarded(m, [&]() { return do_route_mark(m, origin, points, on_device != 0, n, layout, max_range, self_too); });
}

int ufo_b200_route_apply(ufo_b200_map* m, uint32_t first_source, uint32_t n_sources, int last)
{
	return guarded(m, [&]() { return do_route_apply(m, first_source, n_sources, last); });
}

int ufo_b200_ipc_export(void* dev_ptr, void* handle64)
{
	if (!dev_ptr || !handle64) return UFO_B200_E_INVALID;
	static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
	cudaIpcMemHandle_t h;
	if (cudaIpcGetMemHandle(&h, dev_ptr) != cudaSuccess) return UFO_B200_E_CUDA;
	memcpy(handle64, &h, 64);
	return UFO_B200_OK;
}

int ufo_b200_ipc_open(const void* handle64, void** dev_ptr)
{
	if (!handle64 || !dev_ptr) return UFO_B200_E_INVALID;
	cudaIpcMemHandle_t h;
	memcpy(&h, handle64, 64);
	if (cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) return UFO_B200_E_CUDA;
	return UFO_B200_OK;
}

int ufo_b200_ipc_close(void* dev_ptr)
{
	if (!dev_ptr) return UFO_B200_E_INVALID;
	return cudaIpcCloseMemHandle(dev_ptr) == cudaSuccess ? UFO_B200_OK : UFO_B200_E_CUDA;
}

int ufo_b200_enable_change_detection(ufo_b200_map* m, int enable)
{
	if (!m) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		sync_map(m);
		// the mask is allocated by the first enable and kept: switched off, it keeps the recorded set
		m->chg_recording = enable != 0;
		if (enable && !m->chg_mask) {
			alloc_arrays(m, Exists::kChange);
			CK(cudaStreamSynchronize(m->stream));
		}
		m->M.chg_mask = m->chg_recording ? m->chg_mask : nullptr;
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_reset_change_detection(ufo_b200_map* m)
{
	if (!m) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		sync_map(m);
		for_each_pool_array(m, [&](const PoolArray& a) {
			if (a.exists == Exists::kChange && a.buf.get()) a.buf.fill(0, m->stream);
		});
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_changed_codes(ufo_b200_map* m, uint32_t depth, uint64_t* codes, size_t cap, size_t* n)
{
	if (!m || !n) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		sync_map(m);
		*n = 0;
		DeviceMap M = m->M;
		M.chg_mask = m->chg_mask;  // also while recording is switched off
		if (!M.chg_mask || !m->n_bricks) return (int)UFO_B200_OK;
		if (depth > M.g.depth_levels) return (int)UFO_B200_E_INVALID;
		const uint32_t dd = std::min(depth, 4u);
		cudaStream_t s = m->stream;
		Buffer<unsigned long long> d_count, d_codes;
		d_count.resize(1, 0, s);
		const uint32_t grid = (uint32_t)(((size_t)m->n_bricks * 64 + 255) / 256);
		k_changed<<<grid, 256, 0, s>>>(M, m->n_bricks, dd, nullptr, 0, d_count.get());
		unsigned long long cnt = 0;
		CK(cudaMemcpyAsync(&cnt, d_count.get(), 8, cudaMemcpyDeviceToHost, s));
		CK(cudaStreamSynchronize(s));
		std::vector<unsigned long long> h(cnt);
		if (cnt) {
			d_codes.resize(cnt);
			d_count.fill(0, s);
			k_changed<<<grid, 256, 0, s>>>(M, m->n_bricks, dd, d_codes.get(), cnt, d_count.get());
			CK(cudaMemcpyAsync(h.data(), d_codes.get(), cnt * 8, cudaMemcpyDeviceToHost, s));
			CK(cudaStreamSynchronize(s));
		}
		if (depth >= 4) {
			// ancestors above the brick + duplicates: snap to `depth` (with the centre bits) and unique
			const unsigned long long lowmask = depth >= 21 ? ~0ull : ((1ull << (3 * depth)) - 1ull);
			const unsigned long long centre = key_to_code({1u << (depth - 1), 1u << (depth - 1), 1u << (depth - 1)});
			for (auto& c : h) c = (c & ~lowmask) | centre;
			std::sort(h.begin(), h.end());
			h.erase(std::unique(h.begin(), h.end()), h.end());
		}
		*n = h.size();
		if (codes) std::memcpy(codes, h.data(), std::min(cap, h.size()) * 8);
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_write_compressed(ufo_b200_map* m, const double* box6, uint32_t min_depth, int data_only,
                              int acceleration_level, int compression_level, void* buf, size_t cap, size_t* size,
                              size_t* uncompressed_size)
{
	if (!m || !size) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		if (!lz4().ok) {
			m->set_error("liblz4.so.1 not found: compressed output is unavailable");
			return (int)UFO_B200_E_UNSUPPORTED;
		}
		std::vector<uint8_t> raw;
		unsigned long long total = 0;
		int rc = export_image(m, 1, min_depth, box6, false, [&](const void* p, size_t len) {
			const uint8_t* b = static_cast<const uint8_t*>(p);
			raw.insert(raw.end(), b, b + len);
		}, &total);
		if (rc != UFO_B200_OK) return rc;
		std::vector<uint8_t> packed;
		if (!lz4_compress(raw, acceleration_level, compression_level, packed)) {
			m->set_error("LZ4 compression failed");
			return (int)UFO_B200_E_INVALID;
		}
		std::string head;
		if (!data_only) {
			// octree.h:850-860 with "compressed 1"
			char h[512];
			const int hl = snprintf(h, sizeof h,
			                        "# UFOMap file\n# (feel free to add / change comments, but leave the first line as it "
			                        "is!)\n#\nversion 1.0.0\nid %s\nresolution %g\ndepth_levels %u\ncompressed 1\n"
			                        "uncompressed_data_size %d\ndata\n",
			                        m->M.color ? "occupancy_map_color" : "occupancy_map", m->M.g.resolution, m->M.g.depth_levels,
			                        (int)raw.size());
			head.assign(h, (size_t)hl);
		}
		const size_t need = head.size() + packed.size();
		*size = need;
		if (uncompressed_size) *uncompressed_size = raw.size();
		if (buf && cap >= need) {
			std::memcpy(buf, head.data(), head.size());
			std::memcpy(static_cast<uint8_t*>(buf) + head.size(), packed.data(), packed.size());
		}
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_cast_rays(ufo_b200_map* m, const double* origins, const double* directions, size_t n,
                       int ignore_unknown, double max_range, uint32_t depth, uint64_t* codes, uint8_t* hit)
{
	if (!m || (n && (!origins || !directions || !codes || !hit)) || n > 0x7fffffffull) return UFO_B200_E_INVALID;
	if (!n) return UFO_B200_OK;
	return guarded(m, [&]() {
		if (depth > m->M.g.depth_levels) return (int)UFO_B200_E_INVALID;
		CK(cudaSetDevice(m->device));
		sync_map(m);
		cudaStream_t s = m->stream;
		std::vector<double> rays(6 * n);
		for (size_t i = 0; i < n; ++i) {
			for (int k = 0; k < 3; ++k) {
				rays[6 * i + k] = origins[3 * i + k];
				rays[6 * i + 3 + k] = directions[3 * i + k];
			}
		}
		Buffer<double> d_rays;
		Buffer<unsigned long long> d_codes;
		Buffer<uint8_t> d_hit;
		d_rays.resize(rays.size());
		d_codes.resize(n);
		d_hit.resize(n);
		CK(cudaMemcpyAsync(d_rays.get(), rays.data(), rays.size() * 8, cudaMemcpyHostToDevice, s));
		k_cast_rays<<<(uint32_t)((n + 127) / 128), 128, 0, s>>>(m->M, d_rays.get(), (uint32_t)n, ignore_unknown, max_range, depth,
		                                                        d_codes.get(), d_hit.get());
		CK(cudaGetLastError());
		CK(cudaMemcpyAsync(codes, d_codes.get(), n * 8, cudaMemcpyDeviceToHost, s));
		CK(cudaMemcpyAsync(hit, d_hit.get(), n, cudaMemcpyDeviceToHost, s));
		CK(cudaStreamSynchronize(s));
		return (int)UFO_B200_OK;
	});
}

int ufo_b200_export_nodes(ufo_b200_map* m, uint32_t depth, int occupied, int free_space, int unknown, const double* box6,
                          uint64_t* codes, float* logodds, uint8_t* rgb, size_t cap, size_t* n)
{
	if (!m || !n) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		CK(cudaSetDevice(m->device));
		sync_map(m);
		*n = 0;
		if (depth > m->M.g.depth_levels) return (int)UFO_B200_E_INVALID;
		NodeFilter f{};
		f.depth = depth;
		f.occupied = occupied;
		f.free_ = free_space;
		f.unknown = unknown;
		if (box6) {
			f.box.on = 1;
			for (int k = 0; k < 3; ++k) {
				f.box.lo[k] = box6[k] - box6[3 + k];
				f.box.hi[k] = box6[k] + box6[3 + k];
			}
		}
		collect_results(m, codes, logodds, rgb, cap, n, [&](unsigned long long* d_codes, float* d_occ, uint32_t* d_rgb,
		                                                     size_t d_cap, unsigned long long* d_count) {
			if (depth <= 4) {
				const size_t threads = (size_t)m->n_bricks * 64;
				if (threads) k_export_nodes<<<(uint32_t)((threads + 255) / 256), 256, 0, m->stream>>>(m->M, m->n_bricks, f, d_codes, d_occ, d_rgb, d_cap, d_count);
			} else if (m->n_upper) {
				k_export_upper<<<(m->n_upper + 255) / 256, 256, 0, m->stream>>>(m->M, m->n_upper, f, d_codes, d_occ, d_rgb, d_cap, d_count);
			}
		});
		return (int)UFO_B200_OK;
	});
}

}  // extern "C"

namespace
{
struct StreamReader {
	const uint8_t* p;
	size_t n, at = 0;
	bool ok = true;
	bool get(void* out, size_t len)
	{
		if (at + len > n) {
			ok = false;
			std::memset(out, 0, len);
			at = n + 1;
			return false;
		}
		std::memcpy(out, p + at, len);
		at += len;
		return true;
	}
};

struct ImportPlan {
	std::vector<ImportRec> small, bricks, wipe;  // depth <= 2, depth 4, depth >= 5
	const Geometry* g = nullptr;
	ExportBox box{};
	uint32_t P = 4;
	uint64_t budget = 1ull << 20;  // bricks a stream may create through collapsed nodes above the brick level
	bool too_big = false;
};

void import_leaf(ImportPlan& plan, uint64_t code, uint32_t depth, float occ, uint32_t rgb)
{
	const ImportRec r{code, depth, occ, rgb, 0u};
	if (depth <= 2) {
		plan.small.push_back(r);
	} else if (depth == 3) {
		for (uint64_t i = 0; i < 8; ++i) plan.small.push_back(ImportRec{code + (i << 6), 2u, occ, rgb, 0u});
	} else if (depth == 4) {
		plan.bricks.push_back(r);
	} else {
		// existing bricks below the node take the payload; if it is not the default, the bricks that
		// do not exist yet have to be created as well (the value field has no collapsed nodes)
		plan.wipe.push_back(r);
		if (occ != 0.0f || rgb != 0u) {
			const uint64_t nb = depth >= 11 ? ~0ull : 1ull << (3 * (depth - 4));
			if (nb > plan.budget) {
				plan.too_big = true;
				return;
			}
			plan.budget -= nb;
			for (uint64_t i = 0; i < nb; ++i) plan.bricks.push_back(ImportRec{code + (i << 12), 4u, occ, rgb, 0u});
		}
	}
}

void read_payload(StreamReader& in, uint32_t P, float& occ, uint32_t& rgb)
{
	uint8_t b[7] = {0, 0, 0, 0, 0, 0, 0};
	in.get(b, P);
	std::memcpy(&occ, b, 4);
	rgb = P == 7 ? ((uint32_t)b[4] | ((uint32_t)b[5] << 8) | ((uint32_t)b[6] << 16)) : 0u;
}

// readNodesRecurs (occupancy_map_base.h:1403-1456): `code` = first voxel of the node of depth `depth`
void import_rec(ImportPlan& plan, StreamReader& in, uint64_t code, uint32_t depth, const double c[3])
{
	const uint32_t cd = depth - 1;
	const double chs = plan.g->half_size[cd];
	uint8_t children = 0;
	if (!in.get(&children, 1)) return;
	for (uint32_t i = 0; i < 8 && in.ok; ++i) {
		double cc[3];
		child_center(c, chs, i, cc);
		if (!box_hits(plan.box, cc, chs)) continue;
		const uint64_t ccode = code + ((uint64_t)i << (3 * cd));
		if ((children >> i) & 1u) {
			if (1 == cd) {
				for (uint32_t j = 0; j < 8; ++j) {
					double gc[3];
					child_center(cc, plan.g->half_size[0], j, gc);
					if (!box_hits(plan.box, gc, plan.g->half_size[0])) continue;
					float occ;
					uint32_t rgb;
					read_payload(in, plan.P, occ, rgb);
					import_leaf(plan, ccode + j, 0, occ, rgb);
				}
			} else {
				import_rec(plan, in, ccode, cd, cc);
			}
		} else {
			float occ;
			uint32_t rgb;
			read_payload(in, plan.P, occ, rgb);
			import_leaf(plan, ccode, cd, occ, rgb);
		}
	}
}

int import_stream(Map* m, const uint8_t* data, size_t size, const double* box6)
{
	DeviceMap& M = m->M;
	if (M.g.depth_levels < 5) {
		m->set_error("readData needs depth_levels >= 5");
		return UFO_B200_E_UNSUPPORTED;
	}
	if (M.route_world > 1 || M.shard_world > 1) {
		m->set_error("readData on a sharded / routed map is not supported");
		return UFO_B200_E_UNSUPPORTED;
	}
	CK(cudaSetDevice(m->device));
	finalize_scan(m);
	ImportPlan plan;
	plan.g = &M.g;
	plan.P = M.color ? 7 : 4;
	if (box6) {
		plan.box.on = 1;
		for (int k = 0; k < 3; ++k) {
			plan.box.lo[k] = box6[k] - box6[3 + k];
			plan.box.hi[k] = box6[k] + box6[3 + k];
		}
	}
	const double c0[3] = {0.0, 0.0, 0.0};
	if (!box_hits(plan.box, c0, M.g.half_size[M.g.depth_levels])) return UFO_B200_OK;  // no node intersects
	StreamReader in{data, size};
	uint8_t children = 0;
	in.get(&children, 1);
	if (0 == children) {
		float occ;
		uint32_t rgb;
		read_payload(in, plan.P, occ, rgb);
		import_leaf(plan, 0, M.g.depth_levels, occ, rgb);
	} else {
		import_rec(plan, in, 0, M.g.depth_levels, c0);
	}
	if (!in.ok) {
		m->set_error("readData: the node stream is truncated");
		return UFO_B200_E_INVALID;
	}
	if (plan.too_big) {
		m->set_error("readData: a collapsed node above the brick level would expand into more than 2^20 bricks");
		return UFO_B200_E_UNSUPPORTED;
	}
	// the codes of a tree of L levels use 3L bits; the pools must hold the bricks the stream creates
	cudaStream_t s = m->stream;
	const size_t n_small = plan.small.size(), n_bricks = plan.bricks.size(), n_wipe = plan.wipe.size();
	Buffer<ImportRec> d_small, d_bricks, d_wipe;
	if (n_small) {
		d_small.resize(n_small);
		CK(cudaMemcpyAsync(d_small.get(), plan.small.data(), n_small * sizeof(ImportRec), cudaMemcpyHostToDevice, s));
	}
	if (n_bricks) {
		d_bricks.resize(n_bricks);
		CK(cudaMemcpyAsync(d_bricks.get(), plan.bricks.data(), n_bricks * sizeof(ImportRec), cudaMemcpyHostToDevice, s));
	}
	if (n_wipe) {
		d_wipe.resize(n_wipe);
		CK(cudaMemcpyAsync(d_wipe.get(), plan.wipe.data(), n_wipe * sizeof(ImportRec), cudaMemcpyHostToDevice, s));
	}
	for (int attempt = 0;; ++attempt) {
		M.scan_id++;
		if (M.scan_id == 0) M.scan_id = 1;
		M.up_epoch++;
		M.dense = 0;
		M.mask_base = M.miss_mask;
		push_counters(m);
		if (n_wipe && m->n_bricks)
			k_import_wipe<<<(uint32_t)(((size_t)m->n_bricks * 64 + 255) / 256), 256, 0, s>>>(M, m->n_bricks, d_wipe.get(), (uint32_t)n_wipe);
		if (n_bricks) k_import_bricks<<<(uint32_t)std::min<size_t>(n_bricks, (size_t)m->sm_count * 16), 64, 0, s>>>(M, d_bricks.get(), (uint32_t)n_bricks);
		if (n_small) k_import_small<<<m->sm_count * 8, 256, 0, s>>>(M, d_small.get(), (uint32_t)n_small);
		k_import_refresh<<<m->sm_count * 8, 256, 0, s>>>(M);
		if (M.color) k_brick_agg<true><<<m->sm_count * 4, 256, 0, s>>>(M);
		else k_brick_agg<false><<<m->sm_count * 4, 256, 0, s>>>(M);
		launch_upper(m);
		CK(cudaGetLastError());
		CK(cudaMemcpyAsync(m->h_ctr.get(), M.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
		CK(cudaStreamSynchronize(s));
		const uint32_t ov = m->h_ctr->overflow;
		if (!ov) break;
		if (attempt > 16) {
			m->set_error("readData: device pools keep overflowing");
			return UFO_B200_E_NOMEM;
		}
		// writing leaves is idempotent: grow and run the whole import again
		m->n_bricks = std::min(m->h_ctr->n_bricks, M.brick_cap);
		grow_pools(m, ov & 6u, m->h_ctr->n_bricks, m->h_ctr->n_upper);
	}
	m->n_bricks = std::min(m->h_ctr->n_bricks, M.brick_cap);
	m->n_upper = std::min(m->h_ctr->n_upper, M.up_cap);
	return UFO_B200_OK;
}
}  // namespace

extern "C" {

int ufo_b200_read_data(ufo_b200_map* m, const double* box6, const void* data, size_t size, int compressed,
                       size_t uncompressed_size)
{
	if (!m || (!data && size)) return UFO_B200_E_INVALID;
	return guarded(m, [&]() {
		if (!compressed) return import_stream(m, static_cast<const uint8_t*>(data), size, box6);
		if (!lz4().ok) {
			m->set_error("liblz4.so.1 not found: compressed input is unavailable");
			return (int)UFO_B200_E_UNSUPPORTED;
		}
		std::vector<uint8_t> raw(std::max<size_t>(uncompressed_size, 1));
		const int n = lz4().decompress(static_cast<const char*>(data), reinterpret_cast<char*>(raw.data()), (int)size, (int)uncompressed_size);
		if (n < 0) {
			m->set_error("readData: LZ4 decompression failed");
			return (int)UFO_B200_E_INVALID;
		}
		return import_stream(m, raw.data(), (size_t)n, box6);
	});
}

}  // extern "C"






