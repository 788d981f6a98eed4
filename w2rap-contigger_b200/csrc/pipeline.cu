// pipeline.cu — host orchestration of the step-2 path on one B200 and the C ABI over it (include/w2rap_step2.h).
//
// Mirrors buildReadQGraph (paths/long/BuildReadQGraph.cc:1253-1327) stage by stage:
//   createDictOMPRecursive  -> count_stage()      (k_good_len, k_minimizer_map x2, [NCCL exchange], k_count_smem, k_count_region + k_scan_region as
//                                                  fallback, k_insert_solid)
//                           -> select_stage()     (w2rap_step2_build: k_select_tile_counts, scan, k_select_solid over the counts that
//                                                  w2rap_step2_count kept, instead of counting; then the same k_insert_solid)
//   recomputeAdjacencies    -> k_adjacency_dense (sharded: k_adjacency)
//   buildEdges              -> unipath_stage()    (k_links, pointer-jumping list ranking, circles, edge emission, k_backfill_slots)
//   buildHBVFromEdges       -> hbv_stage()        (end keys, radix sort, vertex ids, incidence)
//   path_reads_OMP(+FixPaths)-> path_stage()
// No CPU fallback: without a usable sm_100 device every compute entry point fails with W2RAP_ERR_NO_DEVICE.
#include <algorithm>
#include <cmath>
#include <chrono>
#include <cstdarg>
#include <exception>
#include <map>
#include <mutex>
#include <thread>
#include <unordered_map>

#include <cuda.h>

#include "../../include/w2rap_step2.h"
#include "../../include/w2rap_step2_counts.h"
#include "device_reads.cuh"
#include "count_part.cuh"
#include "kernels.cuh"
#include "shardgraph_kernels.cuh"
#include "nccl_dl.h"
#include "prims.cuh"
#include "slab_freelist.h"
#include "places.cuh"

// behind the opaque handle of w2rap_step2_count / w2rap_step2_build (include/w2rap_step2_counts.h): the k-mers one count kept and
// what a build needs to reproduce a run's counters.  `solid` and `count` are plain cudaMallocAsync allocations on the reads' device,
// not pieces of the device slab, which is leased per call.
struct w2rap_counts {
    const w2rap_device_reads* reads = nullptr;     // the read set counted: a build must pass the same handle ...
    uint64_t n_reads = 0, n_bases = 0;              // ... still holding the same reads
    int device = 0;
    uint32_t min_qual = 0, f0 = 0;                  // quality floor of the count; keep floor (every k-mer seen >= f0 times is kept)
    uint64_t n_kmer_instances = 0, n_distinct = 0, n_kept = 0;     // n_kept: on this rank
    uint64_t hist[101] = {};                        // (whole-job counters: identical on every rank of a sharded count)
    const w2rap_comm* comm = nullptr;               // sharded count: the communicator (null: single GPU), this rank, the world ...
    int world = 1, rank = 0;
    uint32_t logP = 0;                              // ... and the partition count 2^logP: a k-mer is kept on its partition's owner
    ulonglong2* solid = nullptr;                    // n_kept records {w0, w1 | raw ctx}, in the order the reduce emitted them
    uint8_t* count = nullptr;                       // n_kept counts, min(255, occurrences), parallel to `solid`
};

namespace w2r {

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
static thread_local double g_alloc_host_ms = 0;      // host time inside the stream-ordered allocator (this thread = this rank's call)

// Output arrays live in pinned host memory.  cudaMallocHost is slow (it maps and locks pages), so blocks are kept in a
// process-wide pool and reused by later calls: steady-state steps pay no allocation.
struct PinnedPool {
    struct Block { void* p; size_t bytes; bool used; };
    std::mutex mu;
    std::vector<Block> blocks;
    void* acquire(size_t bytes) {
        if (bytes < 64) bytes = 64;
        std::lock_guard<std::mutex> g(mu);
        int best = -1;
        for (size_t i = 0; i < blocks.size(); ++i)
            if (!blocks[i].used && blocks[i].bytes >= bytes && blocks[i].bytes <= 2 * bytes + 4096 && (best < 0 || blocks[i].bytes < blocks[best].bytes)) best = (int)i;
        if (best >= 0) { blocks[best].used = true; return blocks[best].p; }
        void* p = nullptr;
        size_t cap = bytes + bytes / 8;       // a little slack so that slightly larger results of the next step still fit
        cudaError_t e = cudaMallocHost(&p, cap);
        if (e != cudaSuccess) {               // drop idle blocks and retry once
            cudaGetLastError();
            for (auto& b : blocks) if (!b.used && b.p) { cudaFreeHost(b.p); b.p = nullptr; b.bytes = 0; }
            W2R_CUDA(cudaMallocHost(&p, cap));
        }
        blocks.push_back(Block{p, cap, true});
        return p;
    }
    void release(void* p) {
        std::lock_guard<std::mutex> g(mu);
        for (auto& b : blocks) if (b.p == p) { b.used = false; return; }
    }
    static PinnedPool& get() { static PinnedPool* pool = new PinnedPool(); return *pool; }   // leaked on purpose: outlives the CUDA context teardown order
};
struct GraphOwner {
    std::vector<void*> pinned;
    ~GraphOwner() { for (void* p : pinned) PinnedPool::get().release(p); }
};
template <class T>
static T* out_alloc(GraphOwner* o, size_t n) {
    void* p = PinnedPool::get().acquire((n ? n : 1) * sizeof(T));
    o->pinned.push_back(p);
    return (T*)p;
}

static void check_device(int device, Ctx& c) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { cudaGetLastError(); W2R_FAIL(W2RAP_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU path"); }
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
    if (device >= n) W2R_FAIL(W2RAP_ERR_NO_DEVICE, "device %d does not exist (%d visible)", device, n);
    // cudaGetDeviceProperties is slow (it queries everything); three attributes, cached per device, are all that is needed
    static int cached_major[16], cached_sms[16];
    static bool cached[16];
    const int slot = device & 15;
    if (!cached[slot]) {
        int major = 0, minor = 0, sms = 0;
        W2R_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
        W2R_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
        W2R_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        if (major < 10) W2R_FAIL(W2RAP_ERR_NO_DEVICE, "device %d (sm_%d%d) is not sm_100; this library only carries sm_100a code", device, major, minor);
        cached_major[slot] = major; cached_sms[slot] = sms; cached[slot] = true;
    }
    W2R_CUDA(cudaSetDevice(device));
    c.device = device;
    c.sm_count = cached_sms[slot];
    static std::once_flag pool_once[16];
    std::call_once(pool_once[device & 15], [&] {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) { uint64_t thr = ~0ull; cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr); }
    });
}

// ---------------------------------------------------------------- device memory
// Large buffers come from ONE contiguous virtual range per device whose physical backing grows on demand (CUDA virtual memory
// management: cuMemAddressReserve / cuMemCreate / cuMemMap) and is kept between calls.  A free list with coalescing hands out
// pieces of it, lowest address first.  Why not cudaMallocAsync for everything: its pool cannot merge freed blocks that came from
// different growth steps, so a job near the device's capacity (BASELINE config 3: ~60 GB of counting areas freed, then one 60 GB
// pathing dictionary) made the pool unmap and re-map tens of GB on every call — more than a second of host time per step.
// One call at a time holds the slab of a device (SlabLease); everything it allocates is used on its one stream (side streams are
// joined before a buffer is released — the same rule cudaFreeAsync imposes), so host-order reuse is stream-order reuse.  A
// concurrent call on the same device, small buffers (< 1 MB) and W2RAP_NO_SLAB=1 (compute-sanitizer runs: it checks bounds per
// allocation) use cudaMallocAsync.
struct DriverVmm {
    CUresult (*AddressReserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*Create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
    CUresult (*Map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
    CUresult (*SetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
    CUresult (*GetGranularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
    CUresult (*Release)(CUmemGenericAllocationHandle) = nullptr;
    bool ok = false;
    DriverVmm() {
        auto get = [](const char* name, void** fn) {
            cudaDriverEntryPointQueryResult st;
            return cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &st) == cudaSuccess && st == cudaDriverEntryPointSuccess && *fn;
        };
        ok = get("cuMemAddressReserve", (void**)&AddressReserve) && get("cuMemCreate", (void**)&Create) && get("cuMemMap", (void**)&Map) &&
             get("cuMemSetAccess", (void**)&SetAccess) && get("cuMemGetAllocationGranularity", (void**)&GetGranularity) && get("cuMemRelease", (void**)&Release);
        if (!ok) cudaGetLastError();
    }
    static DriverVmm& get() { static DriverVmm* v = new DriverVmm(); return *v; }
};

struct DeviceSlab {
    static constexpr size_t MIN_BYTES = 1u << 20;        // smaller requests stay with cudaMallocAsync
    static constexpr size_t ALIGN = 4096;
    std::mutex lease;                                    // held by the one call that uses the slab
    int device = -1;
    bool disabled = false;
    CUdeviceptr base = 0;
    size_t va_bytes = 0, mapped = 0, gran = 0;
    SlabFreeList fl;                                     // which pieces of [0, mapped) are in use (slab_freelist.h)

    static DeviceSlab& get(int device) { static DeviceSlab* s = new DeviceSlab[16]; return s[device & 15]; }   // leaked on purpose (see PinnedPool)
    bool contains(const void* p) const { return base && (CUdeviceptr)p >= base && (CUdeviceptr)p < base + va_bytes; }
    size_t idle_bytes() const { return mapped - fl.used; }

    bool init(int dev) {
        if (disabled) return false;
        if (base) return true;
        DriverVmm& v = DriverVmm::get();
        static const bool off = getenv("W2RAP_NO_SLAB") != nullptr;
        size_t fr = 0, tot = 0;
        if (off || !v.ok || cudaMemGetInfo(&fr, &tot) != cudaSuccess) { cudaGetLastError(); disabled = true; return false; }
        CUmemAllocationProp prop = {};
        prop.type = CU_MEM_ALLOCATION_TYPE_PINNED; prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE; prop.location.id = dev;
        if (v.GetGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || !gran) { disabled = true; return false; }
        va_bytes = (tot + gran - 1) / gran * gran;
        if (v.AddressReserve(&base, va_bytes, gran, 0, 0) != CUDA_SUCCESS) { base = 0; disabled = true; return false; }
        device = dev;
        return true;
    }
    // physical backing for [mapped, mapped + bytes): one cuMemCreate per growth step
    bool grow(size_t need) {
        DriverVmm& v = DriverVmm::get();
        size_t want = std::max<size_t>(need, 256u << 20);
        want = (want + gran - 1) / gran * gran;
        for (int attempt = 0; attempt < 2; ++attempt) {
            size_t fr = 0, tot = 0;
            if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { cudaGetLastError(); return false; }
            const size_t margin = 512u << 20;            // NCCL, the pool's small buffers, the CUDA context
            size_t can = fr > margin ? (fr - margin) / gran * gran : 0;
            size_t take = std::min(want, can);
            if (take >= (need + gran - 1) / gran * gran && mapped + take <= va_bytes) {
                CUmemAllocationProp prop = {};
                prop.type = CU_MEM_ALLOCATION_TYPE_PINNED; prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE; prop.location.id = device;
                CUmemGenericAllocationHandle h;
                if (v.Create(&h, take, &prop, 0) == CUDA_SUCCESS) {
                    CUmemAccessDesc acc = {};
                    acc.location = prop.location; acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
                    if (v.Map(base + mapped, take, 0, h, 0) == CUDA_SUCCESS && v.SetAccess(base + mapped, take, &acc, 1) == CUDA_SUCCESS) {
                        v.Release(h);                    // the mapping keeps the memory alive
                        fl.add_free(mapped, take);
                        mapped += take;
                        return true;
                    }
                    v.Release(h);
                    return false;
                }
            }
            // memory cached by the stream-ordered pool may be what is missing: give it back and try once more
            cudaMemPool_t pool;
            if (attempt == 0 && cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) { cudaDeviceSynchronize(); cudaMemPoolTrimTo(pool, 0); } else break;
        }
        return false;
    }
    void* acquire(size_t bytes) {
        bytes = (bytes + ALIGN - 1) / ALIGN * ALIGN;
        size_t off = fl.take(bytes);
        if (off == SlabFreeList::NONE) {
            // nothing fits: extend the top (only by what the free range touching it lacks)
            if (!grow(bytes - fl.free_tail(mapped))) return nullptr;
            off = fl.take(bytes);
            if (off == SlabFreeList::NONE) return nullptr;
        }
        return (void*)(base + off);
    }
    void release(void* p) { fl.give_back((size_t)((CUdeviceptr)p - base)); }
};
// one call holds a device's slab from its first buffer to its last; a failed call drains the device before handing it on
struct SlabLease {
    DeviceSlab* slab = nullptr;
    explicit SlabLease(int device) {
        DeviceSlab& s = DeviceSlab::get(device);
        if (s.lease.try_lock()) { if (s.init(device)) slab = &s; else s.lease.unlock(); }
    }
    ~SlabLease() {
        if (!slab) return;
        if (std::uncaught_exceptions() > 0) cudaDeviceSynchronize();
        slab->lease.unlock();
    }
    SlabLease(const SlabLease&) = delete;
    SlabLease& operator=(const SlabLease&) = delete;
};

// device buffer with stream-ordered lifetime: from the leased slab when it is large, else from CUDA's pool (which caches too)
template <class T>
struct SBuf {
    T* p = nullptr;
    size_t n = 0;
    cudaStream_t s = nullptr;
    DeviceSlab* slab = nullptr;
    SBuf() {}
    SBuf(Ctx& c, size_t n_) { alloc(c, n_); }
    SBuf(const SBuf&) = delete;
    SBuf& operator=(const SBuf&) = delete;
    SBuf(SBuf&& o) noexcept : p(o.p), n(o.n), s(o.s), slab(o.slab) { o.p = nullptr; o.n = 0; o.slab = nullptr; }
    SBuf& operator=(SBuf&& o) noexcept { if (this != &o) { release(); p = o.p; n = o.n; s = o.s; slab = o.slab; o.p = nullptr; o.n = 0; o.slab = nullptr; } return *this; }
    ~SBuf() { release(); }
    void alloc(Ctx& c, size_t n_) {
        release();
        s = c.stream; n = n_;
        if (!n) return;
        const double t0 = now_ms();
        const size_t bytes = n * sizeof(T);
        DeviceSlab* sl = (DeviceSlab*)c.slab;
        if (sl && bytes >= DeviceSlab::MIN_BYTES) { p = (T*)sl->acquire(bytes); if (p) slab = sl; }
        cudaError_t e = cudaSuccess;
        if (!p) e = cudaMallocAsync((void**)&p, bytes, s);
        const double dt = now_ms() - t0;
        g_alloc_host_ms += dt;
        if (dt > 20.0 && getenv("W2RAP_TRACE")) fprintf(stderr, "[w2rap] device allocation of %.2f GB took %.1f ms on the host\n", bytes / 1e9, dt);
        W2R_CUDA(e);
    }
    void release() {
        if (p) {
            const double t0 = now_ms();
            if (slab) slab->release(p); else cudaFreeAsync(p, s);
            g_alloc_host_ms += now_ms() - t0;
        }
        p = nullptr; n = 0; slab = nullptr;
    }
    size_t bytes() const { return n * sizeof(T); }
    void zero() { if (n) W2R_CUDA(cudaMemsetAsync(p, 0, bytes(), s)); }
    void fill_ff() { if (n) W2R_CUDA(cudaMemsetAsync(p, 0xff, bytes(), s)); }
};

// what a call may still allocate: free device memory + what the pool and the slab hold idle
static size_t device_budget(const Ctx& c) {
    size_t fr = 0, tot = 0;
    W2R_CUDA(cudaMemGetInfo(&fr, &tot));
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, c.device) == cudaSuccess) {
        uint64_t reserved = 0, used = 0;
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved);
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
        if (reserved > used) fr += (size_t)(reserved - used);
    }
    if (c.slab) fr += ((const DeviceSlab*)c.slab)->idle_bytes();
    return fr;
}

struct StageTimer {
    Ctx& c;
    cudaEvent_t ev[2];
    explicit StageTimer(Ctx& c_) : c(c_) { cudaEventCreate(&ev[0]); cudaEventCreate(&ev[1]); }
    ~StageTimer() { cudaEventDestroy(ev[0]); cudaEventDestroy(ev[1]); }
    void start() { cudaEventRecord(ev[0], c.stream); }
    float stop() { cudaEventRecord(ev[1], c.stream); cudaEventSynchronize(ev[1]); float ms = 0; cudaEventElapsedTime(&ms, ev[0], ev[1]); return ms; }
};

// CUDA-event time of individual kernels without stalling the queue: events are recorded around the launches and read once the
// stream has drained (w2rap_timings.kernel_ms).
struct KernelTimers {
    struct Span { int idx; cudaEvent_t a, b; };
    std::vector<Span> spans;
    cudaStream_t s = nullptr;
    void begin(int idx) { Span sp{idx, nullptr, nullptr}; cudaEventCreate(&sp.a); cudaEventCreate(&sp.b); cudaEventRecord(sp.a, s); spans.push_back(sp); }
    void end() { cudaEventRecord(spans.back().b, s); }
    void resolve(float* kernel_ms) {
        for (Span& sp : spans) {
            float ms = 0;
            if (cudaEventSynchronize(sp.b) == cudaSuccess && cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) kernel_ms[sp.idx] += ms; else cudaGetLastError();
            cudaEventDestroy(sp.a); cudaEventDestroy(sp.b);
        }
        spans.clear();
    }
    ~KernelTimers() { for (Span& sp : spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); } }
};
#define W2R_TIMED(idx, ...) do { kt_.begin(idx); __VA_ARGS__; kt_.end(); } while (0)

static void say(const Ctx& c, const char* fmt, ...) {
    if (!c.verbose) return;
    va_list ap; va_start(ap, fmt); vprintf(fmt, ap); va_end(ap); printf("\n"); fflush(stdout);
}

// ---------------------------------------------------------------- the pipeline
struct Pipeline {
    Ctx c;
    const DeviceReads& dr;
    const w2rap_params& prm;
    w2rap_graph* out;
    GraphOwner* owner;
    std::vector<DumpRec> dump_host;
    KernelTimers kt_;

    // W2RAP_TRACE: wall-clock of the phases (drains the stream at every mark, so the totals of a traced run are not a measurement)
    double trace_t0 = 0;
    void trace_mark(const char* what) {
        static const bool on = getenv("W2RAP_TRACE") != nullptr;
        if (!on) return;
        cudaStreamSynchronize(c.stream);
        const double t = now_ms();
        if (trace_t0 && rank == 0) fprintf(stderr, "[w2rap] %-28s %8.1f ms   (allocator so far %.1f ms)\n", what, t - trace_t0, g_alloc_host_ms);
        trace_t0 = t;
    }

    // persistent device state between stages
    SBuf<uint16_t> good;
    SBuf<SolidSlot> solid_slots;
    SolidTable st{nullptr, 0};
    SBuf<SolidSlot> dense_slots;            // one GPU: the graph stage's nodes (unipath.cuh: DenseNodes), from the dictionary build to emit
    DenseNodes dn{{nullptr, 0}, nullptr, 0};
    uint64_t E = 0, nv = 0, nh = 0;
    SBuf<uint8_t> edge_bases; SBuf<uint64_t> edge_off; SBuf<uint32_t> edge_len;
    SBuf<int32_t> edge_vertices, fwd_xlat, rev_xlat, involution, hleft, hright, from_e, to_e;
    SBuf<uint32_t> hcanon;
    SBuf<uint8_t> from_n, to_n;
    uint64_t edge_bytes = 0;
    int world = 1, rank = 0;            // sharded run: one process per GPU, reads sharded by index, k-mers routed to owners
    ncclComm_t comm = nullptr;

    bool keep_counts = false;                   // w2rap_step2_count: the reduce also writes the count of every solid record
    const w2rap_counts* from_counts = nullptr;  // w2rap_step2_build: the solid records are selected from these instead of counted

    Pipeline(const DeviceReads& dr_, const w2rap_params& p_, w2rap_graph* out_, GraphOwner* ow) : dr(dr_), prm(p_), out(out_), owner(ow) {}

    unsigned grid(uint64_t n, unsigned block, unsigned per_sm = 16) const { return grid_for(c, n, block, per_sm); }

    // ---- createDictOMPRecursive (BuildReadQGraph.cc:1015-1117): partition (map) + L2-resident hash count (reduce), count_part.cuh
    void set_l2_window(void* base, size_t bytes) {
        cudaStreamAttrValue attr;
        memset(&attr, 0, sizeof attr);
        attr.accessPolicyWindow.base_ptr = base;
        attr.accessPolicyWindow.num_bytes = bytes;
        attr.accessPolicyWindow.hitRatio = 1.0f;
        attr.accessPolicyWindow.hitProp = bytes ? cudaAccessPropertyPersisting : cudaAccessPropertyNormal;
        attr.accessPolicyWindow.missProp = bytes ? cudaAccessPropertyStreaming : cudaAccessPropertyNormal;
        if (cudaStreamSetAttribute(c.stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
    }

    // ---- multi-GPU plumbing (NCCL over NVLink/NVSwitch); world == 1 needs none of it
    void nccl_check(ncclResult_t r, const char* what) {
        if (r != ncclSuccess) W2R_FAIL(W2RAP_ERR_CUDA, "NCCL %s failed: %s", what, NcclApi::get().GetErrorString ? NcclApi::get().GetErrorString(r) : "?");
    }
    // element-wise all-reduce of a small host vector of u64 (through a device staging buffer)
    void allreduce_u64(std::vector<unsigned long long>& v, ncclRedOp_t op) {
        if (world == 1) return;
        SBuf<unsigned long long> d(c, v.size());
        W2R_CUDA(cudaMemcpyAsync(d.p, v.data(), v.size() * 8, cudaMemcpyHostToDevice, c.stream));
        nccl_check(NcclApi::get().AllReduce(d.p, d.p, v.size(), ncclUint64, op, comm, c.stream), "all-reduce");
        W2R_CUDA(cudaMemcpyAsync(v.data(), d.p, v.size() * 8, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
    }
    // all-to-all of equal slabs: slab d of `send` goes to rank d, slab s of `recv` comes from rank s (MapReduceEngine's "swizzle",
    // MapReduceEngine.h:337-358, as grouped ncclSend/ncclRecv over NVLink)
    void alltoall_slabs(const void* send, void* recv, size_t slab_bytes) {
        NcclApi& n = NcclApi::get();
        nccl_check(n.GroupStart(), "group start");
        for (int peer = 0; peer < world; ++peer) {
            if (peer == rank) continue;
            nccl_check(n.Send((const char*)send + (size_t)peer * slab_bytes, slab_bytes, ncclUint8, peer, comm, c.stream), "send");
            nccl_check(n.Recv((char*)recv + (size_t)peer * slab_bytes, slab_bytes, ncclUint8, peer, comm, c.stream), "recv");
        }
        nccl_check(n.GroupEnd(), "group end");
        W2R_CUDA(cudaMemcpyAsync((char*)recv + (size_t)rank * slab_bytes, (const char*)send + (size_t)rank * slab_bytes, slab_bytes, cudaMemcpyDeviceToDevice, c.stream));
    }

    // byte-granular all-to-all with per-peer sizes (the minimiser layout: every rank sends each peer exactly the runs of the
    // partitions that peer owns)
    void alltoall_v(const void* send, const std::vector<size_t>& soff, const std::vector<size_t>& scnt, void* recv, const std::vector<size_t>& roff,
                    const std::vector<size_t>& rcnt) {
        NcclApi& n = NcclApi::get();
        nccl_check(n.GroupStart(), "group start");
        for (int peer = 0; peer < world; ++peer) {
            if (peer == rank) continue;
            if (scnt[peer]) nccl_check(n.Send((const char*)send + soff[peer], scnt[peer], ncclUint8, peer, comm, c.stream), "send");
            if (rcnt[peer]) nccl_check(n.Recv((char*)recv + roff[peer], rcnt[peer], ncclUint8, peer, comm, c.stream), "recv");
        }
        nccl_check(n.GroupEnd(), "group end");
        if (scnt[rank]) W2R_CUDA(cudaMemcpyAsync((char*)recv + roff[rank], (const char*)send + soff[rank], scnt[rank], cudaMemcpyDeviceToDevice, c.stream));
    }

    // ---- createDictOMPRecursive (BuildReadQGraph.cc:1000-1108): quality floor, k-mer counting, min-frequency filter, dictionary.
    // map (k_good_len, k_minimizer_map x2 per read batch) -> [NCCL exchange of the records to the partition owners] ->
    // reduce (k_count_smem; k_count_region/k_scan_region for partitions that do not fit shared memory) -> solid records.
    struct Batch { uint64_t first, count; cudaEvent_t ready; };      // reads [first, first+count) with an event to wait for (nullptr = resident)
    struct CountPlan {
        uint32_t logP = 0, npass = 1, nmap = 1, nslab = 1;
        uint64_t P = 1, Pown = 1;
        uint64_t n_inst = 0, n_inst_local = 0;        // upper bounds: whole job / this rank
    };
    // device state of one counting attempt
    struct CountBufs {
        SBuf<SkmRec> recs, xrecs;                      // local record area; sharded: the records this rank owns after the exchange
        SBuf<SkmRec> tmp; SBuf<uint32_t> tpart;        // staging area of the map: records in production order + the partition of each
        SBuf<unsigned long long> tmp_cursor, tmp_range;   // slots handed out; [nmap + 1] staging range of every read batch
        SBuf<uint32_t> part_count, part_kcount, cursor;   // [nmap][P]
        SBuf<uint64_t> part_base, batch_total, batch_ktotal;
        SBuf<unsigned long long> batch_off;            // [nmap + 1]
        SBuf<uint32_t> xcount, xkcount;                // sharded: [world][Pown] records / k-mers of my partitions held by each rank
        SBuf<uint64_t> xbase, xtot, xktot;
        SBuf<unsigned long long> xoff;                 // [world + 1]
    };
    SBuf<unsigned long long> cs_scal;                  // [0] k-mer instances, [1] solid cursor, [2] dump cursor, [4] failed-partition cursor
    SBuf<int> cs_flags;                                // [0] malformed quality vector, [1] record buffer overflow, [2] solid staging overflow
    SBuf<unsigned long long> cs_hist;
    SBuf<CountSlot> cs_region;                         // two L2-resident counting regions (fallback reduce)
    SBuf<DumpRec> cs_dump;
    SBuf<ulonglong2> cs_solid; uint64_t cs_solid_cap = 0;
    SBuf<uint8_t> cs_count;                            // keep_counts: min(255, count) of cs_solid[i], same capacity
    uint64_t cs_R = 0; uint32_t cs_logR = 0;
    bool good_done = false;
    float map_ms = 0, reduce_ms = 0, xchg_ms = 0;
    uint32_t n_groups = 0;
    uint64_t xchg_bytes = 0, xchg_count_bytes = 0, n_records = 0;

    void run_good_len(const Batch& bt) {
        if (bt.ready) W2R_CUDA(cudaStreamWaitEvent(c.stream, bt.ready, 0));
        if (bt.count) W2R_TIMED(W2RAP_KT_GOOD_LEN, W2R_LAUNCH(c, k_good_len, grid(bt.count, 128), 128, 0, dr.view(), bt.first, bt.count, prm.min_qual, good.p, cs_scal.p, cs_flags.p));
    }

    // warps of the map launch over `count` reads that take a staging chunk: each ends the launch holding one partly used chunk
    uint64_t map_chunk_warps(uint64_t count) const { return std::min<uint64_t>(count, (uint64_t)grid(count * 32, 256, MAP_CTAS_PER_SM) * 8); }

    // map: per read batch  quality floor -> counting launch -> scan -> store launch (all queued without a host round trip, so a
    // batch is mapped as soon as it has crossed PCIe).  Returns false if the record area was too small (need = exact size).
    bool map_records(const CountPlan& pl, CountBufs& cb, const std::vector<Batch>& batches, uint32_t pass, uint64_t* need) {
        const ReadsView rv = dr.view();
        const uint64_t P = pl.P;
        cb.cursor.zero(); cb.part_count.zero(); cb.part_kcount.zero();
        W2R_CUDA(cudaMemsetAsync(cb.batch_off.p, 0, sizeof(unsigned long long), c.stream));
        std::vector<Batch> mb = batches;
        if (world > 1) {        // sharded: one map batch (the layout must be by owner rank), after the whole shard has arrived
            if (!good_done) for (const Batch& bt : batches) run_good_len(bt);
            good_done = true;
            mb.assign(1, Batch{0, dr.n, nullptr});
        }
        std::vector<cudaEvent_t> ev(2 * pl.nmap, nullptr);                 // the map launches are timed without stalling the queue
        struct EvGuard { std::vector<cudaEvent_t>& v; ~EvGuard() { for (cudaEvent_t e : v) if (e) cudaEventDestroy(e); } } evg{ev};
        W2R_CUDA(cudaMemsetAsync(cb.tmp_cursor.p, 0, 8, c.stream));
        W2R_CUDA(cudaMemsetAsync(cb.tpart.p, 0xff, cb.tpart.bytes(), c.stream));      // NIL: unused staging slot
        for (uint32_t bi = 0; bi < pl.nmap; ++bi) {
            const Batch& bt = mb[bi];
            MiniParams mp{pl.logP, pl.npass, pass, cb.part_count.p + bi * P, cb.part_kcount.p + bi * P, cb.tmp.p, cb.tpart.p, cb.tmp_cursor.p, cb.tmp.n, cs_flags.p + 1};
            ScatterParams sp{cb.tmp.p, cb.tpart.p, cb.tmp_range.p + bi, cb.part_base.p + bi * P, cb.cursor.p + bi * P, cb.recs.p, cb.batch_off.p + bi, cb.recs.n, cb.tmp.n, cs_flags.p + 1};
            if (!good_done) run_good_len(bt);
            W2R_CUDA(cudaEventCreate(&ev[2 * bi])); W2R_CUDA(cudaEventCreate(&ev[2 * bi + 1]));
            W2R_CUDA(cudaEventRecord(ev[2 * bi], c.stream));
            W2R_LAUNCH(c, k_copy_scalar, 1, 1, 0, (const unsigned long long*)cb.tmp_cursor.p, cb.tmp_range.p + bi);
            if (bt.count && pl.n_inst_local) W2R_TIMED(W2RAP_KT_MAP, W2R_LAUNCH(c, k_minimizer_map, grid(bt.count * 32, 256, MAP_CTAS_PER_SM), 256, 0, rv, bt.first, bt.count, good.p, mp));
            W2R_LAUNCH(c, k_copy_scalar, 1, 1, 0, (const unsigned long long*)cb.tmp_cursor.p, cb.tmp_range.p + bi + 1);
            exclusive_scan<uint32_t, uint64_t>(c, cb.part_count.p + bi * P, P, cb.part_base.p + bi * P, cb.batch_total.p + bi);
            W2R_LAUNCH(c, k_next_batch_off, 1, 1, 0, cb.batch_off.p + bi, cb.batch_total.p + bi);
            if (bt.count && pl.n_inst_local) { W2R_TIMED(W2RAP_KT_SCATTER, W2R_LAUNCH(c, k_scatter_records, (unsigned)(c.sm_count * 8), 256, 0, sp)); c.count_launches++; }
            W2R_CUDA(cudaEventRecord(ev[2 * bi + 1], c.stream));
        }
        good_done = true;
        unsigned long long total = 0, staged = 0;
        W2R_CUDA(cudaMemcpyAsync(&total, cb.batch_off.p + pl.nmap, 8, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaMemcpyAsync(&staged, cb.tmp_cursor.p, 8, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        for (uint32_t bi = 0; bi < pl.nmap; ++bi) { float ms = 0; cudaEventElapsedTime(&ms, ev[2 * bi], ev[2 * bi + 1]); map_ms += ms; }
        if (d2h_scalar(c, cs_flags.p)) W2R_FAIL(W2RAP_ERR_BAD_ARG, "a read's quality vector does not have one quality per base");
        n_records += total;
        *need = std::max(total, staged);       // (the staging area also holds the unused ends of the warps' chunks)
        std::vector<unsigned long long> of = {(unsigned long long)d2h_scalar(c, cs_flags.p + 1)};
        allreduce_u64(of, ncclMax);               // every rank must take the same branch
        if (of[0]) { W2R_CUDA(cudaMemsetAsync(cs_flags.p + 1, 0, sizeof(int), c.stream)); return false; }
        return true;
    }

    // sharded: route every record to the rank that owns its partition.  The local area is laid out by partition = by owner, so
    // "everything rank d owns" is one contiguous piece: exchange the per-partition counts, scan them into the receive layout,
    // then one grouped ncclSend/ncclRecv per peer (MapReduceEngine's swizzle, MapReduceEngine.h:337-358, over NVLink).
    void exchange_records(const CountPlan& pl, CountBufs& cb) {
        EventTimer kt(c.stream);
        kt.start();
        const uint64_t Pown = pl.Pown;
        alltoall_slabs(cb.part_count.p, cb.xcount.p, Pown * sizeof(uint32_t));          // xcount[s][q] = records of my partition q held by rank s
        alltoall_slabs(cb.part_kcount.p, cb.xkcount.p, Pown * sizeof(uint32_t));
        W2R_CUDA(cudaMemsetAsync(cb.xoff.p, 0, sizeof(unsigned long long), c.stream));
        for (int sidx = 0; sidx < world; ++sidx) {
            exclusive_scan<uint32_t, uint64_t>(c, cb.xcount.p + (uint64_t)sidx * Pown, Pown, cb.xbase.p + (uint64_t)sidx * Pown, cb.xtot.p + sidx);
            W2R_LAUNCH(c, k_next_batch_off, 1, 1, 0, cb.xoff.p + sidx, cb.xtot.p + sidx);
        }
        std::vector<uint64_t> sbeg(world + 1, 0), rtot(world, 0);
        for (int d = 0; d < world; ++d) W2R_CUDA(cudaMemcpyAsync(&sbeg[d], cb.part_base.p + (uint64_t)d * Pown, 8, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaMemcpyAsync(&sbeg[world], cb.batch_total.p, 8, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaMemcpyAsync(rtot.data(), cb.xtot.p, world * 8, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        std::vector<size_t> soff(world), scnt(world), roff(world), rcnt(world);
        size_t racc = 0;
        for (int d = 0; d < world; ++d) {
            soff[d] = sbeg[d] * sizeof(SkmRec); scnt[d] = (sbeg[d + 1] - sbeg[d]) * sizeof(SkmRec);
            roff[d] = racc * sizeof(SkmRec); rcnt[d] = rtot[d] * sizeof(SkmRec); racc += rtot[d];
            if (d != rank) { xchg_bytes += scnt[d]; xchg_count_bytes += scnt[d]; }
        }
        cb.xrecs.alloc(c, racc + 1);
        alltoall_v(cb.recs.p, soff, scnt, cb.xrecs.p, roff, rcnt);
        xchg_ms += kt.stop();
    }

    // reduce: what this rank counts is `nslab` runs per owned partition (read batches on one GPU, source ranks when sharded)
    void reduce_records(const CountPlan& pl, const SkmRec* xrecs, const uint32_t* xcur, const uint32_t* xkcur, RunView runs, cudaStream_t s2, cudaEvent_t ev_fork, cudaEvent_t ev_join) {
        const uint64_t Pown = pl.Pown, R = cs_R;
        const uint32_t nslab = pl.nslab;
        EventTimer kt(c.stream);
        kt.start();
        SBuf<uint32_t> failed(c, Pown);
        W2R_CUDA(cudaMemsetAsync(cs_scal.p + 4, 0, 8, c.stream));
        // (a per-device attribute: set on every call — ranks driven from threads of one process each have their own device)
        const size_t stage_bytes = (size_t)2 * SKM_CHUNK * sizeof(SkmRec);
        void (*const count_smem)(SmemCountParams) = keep_counts ? k_count_smem<true> : k_count_smem<false>;
        W2R_CUDA(cudaFuncSetAttribute(count_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((20u << SMEM_LOG_SLOTS_MAX) + stage_bytes)));
        // the table_slots test hook shrinks the shared-memory table as well, so that partitions really take the fallback path
        const uint32_t log_slots = prm.table_slots ? (uint32_t)std::max(2, std::min((int)SMEM_LOG_SLOTS_MAX, (int)cs_logR - 6)) : SMEM_LOG_SLOTS_MAX;
        SmemCountParams sc{xrecs, xcur, runs.part_base, runs.slab_off, nslab, (uint32_t)Pown, prm.min_freq, cs_hist.p, cs_solid.p, cs_scal.p + 1, cs_solid_cap, cs_flags.p + 2,
                           prm.dump_kmers == 2 ? cs_dump.p : nullptr, cs_scal.p + 2, failed.p, cs_scal.p + 4, log_slots, cs_count.p};
        kt_.begin(W2RAP_KT_REDUCE);
        count_smem<<<(unsigned)std::min<uint64_t>(Pown, (uint64_t)c.sm_count), 1024, ((size_t)20u << log_slots) + stage_bytes, c.stream>>>(sc); c.launches++; ++n_groups;
        kt_.end();
        W2R_CUDA(cudaGetLastError());
        const uint64_t nfail = d2h_scalar(c, cs_scal.p + 4);
        if (nfail) {
            say(c, "%llu of %llu k-mer partitions did not fit shared memory; counting them through the L2 region", (unsigned long long)nfail, (unsigned long long)Pown);
            std::vector<uint32_t> fl(nfail);
            W2R_CUDA(cudaMemcpyAsync(fl.data(), failed.p, nfail * 4, cudaMemcpyDeviceToHost, c.stream));
            // per owned partition: largest run in records (sizes the grid) and k-mer instances (bounds its distinct k-mers)
            std::vector<uint32_t> raw((size_t)nslab * Pown), rawk((size_t)nslab * Pown);
            W2R_CUDA(cudaMemcpyAsync(raw.data(), xcur, raw.size() * 4, cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaMemcpyAsync(rawk.data(), xkcur, rawk.size() * 4, cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));
            std::vector<uint32_t> sizes(Pown, 0);
            std::vector<uint64_t> totals(Pown, 0);
            for (uint32_t sidx = 0; sidx < nslab; ++sidx)
                for (uint64_t q = 0; q < Pown; ++q) { sizes[q] = std::max(sizes[q], raw[sidx * Pown + q]); totals[q] += rawk[sidx * Pown + q]; }
            // the persisting carve-out is taken from the normal L2, which the map needs for write combining: hold it only while it is used
            if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, std::min<size_t>(2 * R * sizeof(CountSlot), 80u << 20)) != cudaSuccess) cudaGetLastError();
            set_l2_window(cs_region.p, 2 * R * sizeof(CountSlot));
            {   // the second stream gets the same L2 window
                cudaStreamAttrValue attr; memset(&attr, 0, sizeof attr);
                attr.accessPolicyWindow.base_ptr = cs_region.p; attr.accessPolicyWindow.num_bytes = 2 * R * sizeof(CountSlot);
                attr.accessPolicyWindow.hitRatio = 1.0f; attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting; attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
                if (cudaStreamSetAttribute(s2, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
            }
            SBuf<int> gflag(c, nfail + 1); gflag.zero();
            uint32_t group_parity = 0;
            auto fork = [&] { W2R_CUDA(cudaEventRecord(ev_fork, c.stream)); W2R_CUDA(cudaStreamWaitEvent(s2, ev_fork, 0)); };
            auto join = [&] { W2R_CUDA(cudaEventRecord(ev_join, s2)); W2R_CUDA(cudaStreamWaitEvent(c.stream, ev_join, 0)); };
            // entries [i0, i0+g) of the failed list go through one counting region together (two regions on two streams alternate)
            auto run_group = [&](uint32_t i0, uint32_t g, uint32_t sub_mask, uint32_t sub_id, int* flag) {
                ++n_groups;
                uint32_t mxg = 0;
                for (uint32_t q = i0; q < i0 + g; ++q) mxg = std::max(mxg, sizes[fl[q]]);
                cudaStream_t gs = (group_parity & 1u) ? s2 : c.stream;
                CountSlot* greg = cs_region.p + ((group_parity & 1u) ? R : 0);
                ++group_parity;
                if (mxg) {
                    RegionParams rp{greg, cs_logR, sub_mask, sub_id, flag};
                    RunView rv2 = runs;
                    rv2.plist = failed.p;
                    dim3 gr(std::max(1u, std::min<unsigned>((mxg + 7) / 8, (unsigned)(c.sm_count * 8 / std::max(1u, std::min(g * nslab, 8u))))), g * nslab);
                    k_count_region<<<gr, 256, 0, gs>>>(xrecs, xcur, i0, g, rv2, rp); c.launches++;
                    W2R_CUDA(cudaGetLastError());
                }
                ScanParams sp{greg, R, prm.min_freq, cs_hist.p, cs_solid.p, cs_scal.p + 1, cs_solid_cap, prm.dump_kmers == 2 ? cs_dump.p : nullptr, cs_scal.p + 2, flag, cs_flags.p + 2, cs_count.p};
                k_scan_region<<<grid(R, 256, 4), 256, 0, gs>>>(sp); c.launches++;
                W2R_CUDA(cudaGetLastError());
            };
            // in bulk: as many listed partitions per region pass as fit it even if every k-mer were distinct (load <= 0.6), no host
            // round trip per group; a group that overflows all the same is redone partition by partition below
            std::vector<std::pair<uint32_t, uint32_t>> lgroups;        // (offset into fl, count)
            const uint32_t gmax = std::max(1u, 4000u / nslab);          // gridDim.y = g * nslab <= 65535
            for (size_t i0 = 0; i0 < fl.size();) {
                uint64_t acc = 0; size_t j = i0;
                while (j < fl.size() && j - i0 < gmax && (j == i0 || (double)(acc + totals[fl[j]]) <= 0.6 * (double)R)) { acc += totals[fl[j]]; ++j; }
                lgroups.push_back({(uint32_t)i0, (uint32_t)(j - i0)});
                i0 = j;
            }
            if (lgroups.size() > nfail) W2R_FAIL(W2RAP_ERR_INTERNAL, "more fallback groups than failed partitions");
            fork();
            for (size_t gi = 0; gi < lgroups.size(); ++gi) run_group(lgroups[gi].first, lgroups[gi].second, 0, 0, gflag.p + gi);
            join();
            std::vector<int> lgf(lgroups.size());
            W2R_CUDA(cudaMemcpyAsync(lgf.data(), gflag.p, lgroups.size() * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));
            int* one_flag = gflag.p + nfail;
            for (size_t gi = 0; gi < lgroups.size(); ++gi) {
                if (!lgf[gi]) continue;
                // the group did not fit together: its partitions one by one, and a partition that still fails in hash sub-ranges
                for (uint32_t k = lgroups[gi].first; k < lgroups[gi].first + lgroups[gi].second; ++k) {
                    unsigned long long snapshot[2];
                    std::vector<unsigned long long> hist_snapshot(104);
                    W2R_CUDA(cudaMemcpyAsync(snapshot, cs_scal.p + 1, 16, cudaMemcpyDeviceToHost, c.stream));
                    W2R_CUDA(cudaMemcpyAsync(hist_snapshot.data(), cs_hist.p, 104 * 8, cudaMemcpyDeviceToHost, c.stream));
                    W2R_CUDA(cudaMemsetAsync(one_flag, 0, sizeof(int), c.stream));
                    fork(); run_group(k, 1, 0, 0, one_flag); join();
                    if (!d2h_scalar(c, one_flag)) continue;
                    for (uint32_t S = 2;; S *= 2) {
                        if (S > 4096) W2R_FAIL(W2RAP_ERR_INTERNAL, "a k-mer partition does not fit the counting region even in 4096 hash sub-ranges");
                        bool ok = true;
                        for (uint32_t sid = 0; sid < S && ok; ++sid) {
                            W2R_CUDA(cudaMemsetAsync(one_flag, 0, sizeof(int), c.stream));
                            fork(); run_group(k, 1, S - 1, sid, one_flag); join();
                            if (d2h_scalar(c, one_flag)) ok = false;
                        }
                        if (ok) break;
                        // roll back what the successful sub-ranges of this split emitted, then split finer (restoring the solid cursor is
                        // enough for cs_count too: the counts are written at the same positions as the records and get overwritten alike)
                        W2R_CUDA(cudaMemcpyAsync(cs_scal.p + 1, snapshot, 16, cudaMemcpyHostToDevice, c.stream));
                        W2R_CUDA(cudaMemcpyAsync(cs_hist.p, hist_snapshot.data(), 104 * 8, cudaMemcpyHostToDevice, c.stream));
                        W2R_CUDA(cudaStreamSynchronize(c.stream));
                    }
                }
            }
            set_l2_window(nullptr, 0);
            W2R_CUDA(cudaStreamSynchronize(c.stream));
            if (cudaCtxResetPersistingL2Cache() != cudaSuccess) cudaGetLastError();
            if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0) != cudaSuccess) cudaGetLastError();
        }
        reduce_ms += kt.stop();
    }

    void count_stage() {
        good.alloc(c, dr.n);
        cs_scal.alloc(c, 8); cs_scal.zero();
        cs_flags.alloc(c, 4); cs_flags.zero();
        cs_hist.alloc(c, 104); cs_hist.zero();
        CountPlan pl;
        // Everything is sized from an upper bound of the instance count that needs no qualities (sum of len-59), so that the
        // quality floor + map of the first read batch can start while later batches are still crossing PCIe.
        pl.n_inst_local = dr.n_inst_upper;
        std::vector<unsigned long long> agg = {pl.n_inst_local};
        allreduce_u64(agg, ncclSum);
        pl.n_inst = agg[0];
        std::vector<Batch> batches;
        if (!dr.batch_ready.empty()) for (size_t b = 0; b < dr.batch_ready.size(); ++b) batches.push_back(Batch{dr.batch_first[b], dr.batch_first[b + 1] - dr.batch_first[b], dr.batch_ready[b]});
        else batches.push_back(Batch{0, dr.n, nullptr});

        // fallback region: 1 Mi slots x 32 B = 32 MB of the 126 MB L2, twice (smaller for tiny inputs / the test hook)
        cs_logR = 20;
        while (cs_logR > 8 && (1ull << (cs_logR - 1)) >= 2 * pl.n_inst + 64) --cs_logR;
        if (prm.table_slots) { cs_logR = 6; while ((2ull << cs_logR) <= prm.table_slots && cs_logR < 24) ++cs_logR; }
        cs_R = 1ull << cs_logR;
        // FINE partitions keyed by minimiser, each small enough for one CTA to count in shared memory: ~24 k k-mer instances
        // (measured, config 2, 8192-slot table).  Rank r owns the contiguous partition range [r*P/world, (r+1)*P/world).
        static const double fine_recs = getenv("W2RAP_FINE_RECS") ? atof(getenv("W2RAP_FINE_RECS")) : 24000.0;
        while (((double)pl.n_inst / (double)(1ull << pl.logP) > fine_recs || (1ull << pl.logP) < (uint64_t)world) && pl.logP < 22) ++pl.logP;
        pl.P = 1ull << pl.logP; pl.Pown = pl.P / world;
        count_logP_ = pl.logP;
        pl.nmap = world > 1 ? 1u : (uint32_t)batches.size();
        pl.nslab = world > 1 ? (uint32_t)world : pl.nmap;
        if (pl.nslab > SMEM_MAX_BATCH) W2R_FAIL(W2RAP_ERR_INTERNAL, "more record runs per partition than the reduce kernel handles");
        if (prm.dump_kmers == 2 && world > 1) W2R_FAIL(W2RAP_ERR_BAD_ARG, "dump level 2 is a single-GPU test hook");
        const size_t budget = (size_t)(device_budget(c) * 0.80);
        cs_region.alloc(c, 2 * cs_R);
        cs_dump.alloc(c, prm.dump_kmers == 2 ? pl.n_inst : 0);
        W2R_LAUNCH(c, k_init_count_table, grid(4 * cs_R, 256), 256, 0, cs_region.p, 2 * cs_R);
        cudaStream_t s2 = nullptr;
        W2R_CUDA(cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
        struct StreamGuard { cudaStream_t s; ~StreamGuard() { if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); } } } s2_guard{s2};
        cudaEvent_t ev_fork, ev_join;
        cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming); cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming);
        struct EventGuard { cudaEvent_t a, b; ~EventGuard() { cudaEventDestroy(a); cudaEventDestroy(b); } } ev_guard{ev_fork, ev_join};

        // Records per k-mer instance: ~1/13 on 250-base reads; short reads approach 1.  The area is sized from an estimate and, if
        // the store launch reports an overflow, re-sized to the exact need the counting launch computed.
        // Expected: one record per read, one per minimiser change (2 / (window + 1) per k-mer for a random order) and one per cut at
        // 32 k-mers (1/32 at most): 1 + 0.074 n for a read of n k-mers — 15.1 for n = 191, measured 14.7.  +15 % margin.
        std::vector<unsigned long long> rk = {dr.n_kreads};
        allreduce_u64(rk, ncclSum);
        double rec_per_inst = pl.n_inst ? std::min(1.0, 1.15 * ((double)rk[0] + 0.074 * (double)pl.n_inst) / (double)pl.n_inst) : 1.0;
        uint64_t need_exact = 0;
        pl.npass = prm.force_passes ? prm.force_passes : 1u;
        for (int attempt = 0;; ++attempt) {
            if (attempt > 12) W2R_FAIL(W2RAP_ERR_INTERNAL, "k-mer partitioning did not converge");
            const uint64_t P = pl.P, Pown = pl.Pown;
            // with several passes the k-mer space is split by minimiser hash: allow for uneven passes
            const size_t local_recs = std::max<uint64_t>(need_exact + need_exact / 64, (uint64_t)((double)pl.n_inst_local * rec_per_inst / pl.npass * (pl.npass > 1 ? 1.25 : 1.0))) + 1024;
            const size_t solid_est = (size_t)((double)pl.n_inst / world / pl.npass / std::max<uint32_t>(1, prm.min_freq) * 1.3) * sizeof(ulonglong2);
            const size_t rec_bytes = (local_recs * 2 + local_recs / 8 + (world > 1 ? (size_t)((double)pl.n_inst * rec_per_inst / world / pl.npass * 1.25) : 0)) * (sizeof(SkmRec) + 4);
            std::vector<unsigned long long> too_big = {(rec_bytes + solid_est + cs_dump.bytes() + (64u << 20) > budget) ? 1ull : 0ull};
            allreduce_u64(too_big, ncclMax);                     // every rank must run the same number of passes
            if (too_big[0] && !prm.force_passes) {
                if (pl.npass >= 4096) W2R_FAIL(W2RAP_ERR_OOM, "not enough device memory for the k-mer records even in 4096 passes");
                pl.npass *= 2; --attempt; continue;              // (more passes are not a failed attempt)
            }
            CountBufs cb;
            // staging: the same records plus the unused ends of the chunks the warps reserve, one per warp in every map launch (one
            // launch per read batch)
            uint64_t chunk_warps = 0;
            if (world > 1) chunk_warps = map_chunk_warps(dr.n);
            else for (const Batch& bt : batches) chunk_warps += map_chunk_warps(bt.count);
            const size_t stage_recs = local_recs + local_recs / 8 + chunk_warps * MAP_CHUNK;
            cb.tmp_cursor.alloc(c, 1); cb.tmp_range.alloc(c, pl.nmap + 1);
            cb.part_count.alloc(c, pl.nmap * P); cb.part_kcount.alloc(c, pl.nmap * P); cb.cursor.alloc(c, pl.nmap * P);
            cb.part_base.alloc(c, pl.nmap * P); cb.batch_total.alloc(c, pl.nmap); cb.batch_ktotal.alloc(c, pl.nmap);
            cb.batch_off.alloc(c, pl.nmap + 1);
            if (world > 1) {
                cb.xcount.alloc(c, world * Pown); cb.xkcount.alloc(c, world * Pown); cb.xbase.alloc(c, world * Pown);
                cb.xtot.alloc(c, world); cb.xktot.alloc(c, world); cb.xoff.alloc(c, world + 1);
            }
            bool retry = false;
            W2R_CUDA(cudaMemsetAsync(cs_scal.p + 1, 0, 16, c.stream));       // solid cursor, dump cursor
            cs_hist.zero();
            n_groups = 0;
            uint64_t solid_used = 0;
            for (uint32_t pass = 0; pass < pl.npass && !retry; ++pass) {
                uint64_t need = 0;
                // the big areas live only as long as they are needed (a 1 Gbp job runs within ~25 % of the device's memory of the
                // limit, and a pool that has to re-map memory on every step costs hundreds of milliseconds)
                cb.recs.alloc(c, local_recs);
                cb.tmp.alloc(c, stage_recs); cb.tpart.alloc(c, stage_recs);
                trace_mark("count: buffers");
                const bool mapped = map_records(pl, cb, batches, pass, &need);
                trace_mark("count: map+scatter");
                cb.tmp.release(); cb.tpart.release();
                if (!mapped) {
                    std::vector<unsigned long long> nd = {need};
                    allreduce_u64(nd, ncclMax);
                    need_exact = std::max<uint64_t>(need_exact, nd[0]);
                    retry = true; break;
                }
                if (world > 1) { exchange_records(pl, cb); cb.recs.release(); }      // (the local area is dead once its records are with their owners)
                trace_mark("count: exchange");
                const uint32_t* xcur = world > 1 ? cb.xcount.p : cb.part_count.p;
                const uint32_t* xkcur = world > 1 ? cb.xkcount.p : cb.part_kcount.p;
                const SkmRec* xrecs = world > 1 ? cb.xrecs.p : cb.recs.p;
                RunView runs = world > 1 ? RunView{cb.xbase.p, cb.xoff.p, Pown, nullptr} : RunView{cb.part_base.p, cb.batch_off.p, Pown, nullptr};
                {   // staging for this pass's solid records: each needs >= min_freq of the k-mer instances this rank reduces
                    SBuf<uint64_t> ktot(c, pl.nslab), kscan(c, Pown);
                    for (uint32_t sidx = 0; sidx < pl.nslab; ++sidx) exclusive_scan<uint32_t, uint64_t>(c, xkcur + (uint64_t)sidx * Pown, Pown, kscan.p, ktot.p + sidx);
                    std::vector<uint64_t> kt_h(pl.nslab);
                    W2R_CUDA(cudaMemcpyAsync(kt_h.data(), ktot.p, pl.nslab * 8, cudaMemcpyDeviceToHost, c.stream));
                    W2R_CUDA(cudaStreamSynchronize(c.stream));
                    uint64_t owned = 0;
                    for (uint64_t v : kt_h) owned += v;
                    const uint64_t want = solid_used + owned / std::max<uint32_t>(1, prm.min_freq) + 1024;
                    if (want > cs_solid_cap) {
                        SBuf<ulonglong2> bigger(c, want + want / 4);
                        if (solid_used) W2R_CUDA(cudaMemcpyAsync(bigger.p, cs_solid.p, solid_used * sizeof(ulonglong2), cudaMemcpyDeviceToDevice, c.stream));
                        cs_solid = std::move(bigger);
                        cs_solid_cap = cs_solid.n;
                        if (keep_counts) {           // the parallel count array grows with it, and keeps what earlier passes wrote
                            SBuf<uint8_t> bigger_count(c, cs_solid_cap);
                            if (solid_used) W2R_CUDA(cudaMemcpyAsync(bigger_count.p, cs_count.p, solid_used, cudaMemcpyDeviceToDevice, c.stream));
                            cs_count = std::move(bigger_count);
                        }
                    }
                }
                trace_mark("count: solid staging");
                reduce_records(pl, xrecs, xcur, xkcur, runs, s2, ev_fork, ev_join);
                trace_mark("count: reduce");
                solid_used = d2h_scalar(c, cs_scal.p + 1);
                if (world > 1) cb.xrecs.release();
            }
            if (retry) continue;
            if (d2h_scalar(c, cs_flags.p + 2)) W2R_FAIL(W2RAP_ERR_INTERNAL, "solid staging buffer overflow");
            break;
        }
        {   // the exact instance count of the whole job (the bound above only sized buffers)
            std::vector<unsigned long long> exact = {(unsigned long long)d2h_scalar(c, cs_scal.p)};
            allreduce_u64(exact, ncclSum);
            out->n_kmer_instances = exact[0];
            say(c, "%llu k-mer instances in quality-floored reads", exact[0]);
        }
        out->timings.count_kernel_ms = map_ms;
        out->timings.region_ms = reduce_ms;
        out->timings.exchange_ms = xchg_ms;
        out->timings.count_passes = n_groups;
        std::vector<unsigned long long> hh(104);
        W2R_CUDA(cudaMemcpyAsync(hh.data(), cs_hist.p, 104 * 8, cudaMemcpyDeviceToHost, c.stream));
        unsigned long long cursors[2];
        W2R_CUDA(cudaMemcpyAsync(cursors, cs_scal.p + 1, 16, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        allreduce_u64(hh, ncclSum);                          // histogram of the whole job
        uint64_t n_distinct = 0;
        for (int i = 1; i <= 100; ++i) { out->hist[i] = hh[i]; n_distinct += hh[i]; }
        const uint64_t n_solid_local = cursors[0];
        if (prm.dump_kmers == 2 && cursors[1]) {
            dump_host.resize(cursors[1]);
            W2R_CUDA(cudaMemcpyAsync(dump_host.data(), cs_dump.p, cursors[1] * sizeof(DumpRec), cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));
        }
        cs_region.release(); cs_dump.release();
        n_solid_local_ = n_solid_local; n_distinct_ = n_distinct;
    }

    // w2rap_step2_build: instead of counting, the solid records are the kept records (w2rap_step2_count) seen >= min_freq times,
    // selected in the order the reduce emitted them (k_select_solid); the counters of the count are the run's counters
    void select_stage() {
        const w2rap_counts& h = *from_counts;
        out->n_kmer_instances = h.n_kmer_instances;
        for (int i = 0; i <= 100; ++i) out->hist[i] = h.hist[i];
        n_distinct_ = h.n_distinct;
        count_logP_ = h.logP;                   // sharded: the graph stage finds a k-mer's owner by the count's partition layout
        n_solid_local_ = 0;
        cs_solid.alloc(c, h.n_kept);
        if (!h.n_kept) return;
        const uint64_t tiles = (h.n_kept + SCAN_TILE - 1) / SCAN_TILE;
        SBuf<uint32_t> tile_n(c, tiles);
        SBuf<uint64_t> tile_base(c, tiles), total(c, 1);
        W2R_LAUNCH(c, k_select_tile_counts, (unsigned)tiles, SCAN_THREADS, 0, (const uint8_t*)h.count, h.n_kept, prm.min_freq, tile_n.p);
        exclusive_scan<uint32_t, uint64_t>(c, tile_n.p, tiles, tile_base.p, total.p);
        W2R_LAUNCH(c, k_select_solid, (unsigned)tiles, SCAN_THREADS, 0, (const ulonglong2*)h.solid, (const uint8_t*)h.count, h.n_kept, prm.min_freq,
                   (const uint64_t*)tile_base.p, cs_solid.p);
        n_solid_local_ = d2h_scalar(c, total.p);
    }

    // the pathing filter (kmer.cuh: PathDict): W slices of path_slice_words words, zeroed; its bits are set while the dictionary is built
    void alloc_path_filter(uint64_t n_solid) {
        path_slice_words = 0;
        path_bloom.release();
        if (n_solid < 4096 || !prm.want_paths) return;
        // ~1.5 bytes per key (false positives ~4 %), at least 4 KB, at most 192 MB unless the dictionary is so large that a capped
        // filter would pass everything (measured at 1.44 G keys with 192 MB: every screened position probed the dictionary)
        constexpr uint64_t PATH_FILTER_CAP = 192ull << 20;
        const uint64_t cap = std::max<uint64_t>(PATH_FILTER_CAP, std::min<uint64_t>(n_solid + n_solid / 2, 8ull << 30));
        const uint64_t bytes = std::min<uint64_t>(cap, std::max<uint64_t>(4096, n_solid * 2));
        path_slice_words = (uint32_t)std::max<uint64_t>(64, bytes / 4 / world);
        path_bloom.alloc(c, (size_t)path_slice_words * world);
        path_bloom.zero();
    }

    // One GPU: the dictionary (kmers/ReadPather.h:176-349) as an open-addressing table over all solid k-mers.  Sharded: every rank keeps
    // the solid k-mers it counted; graph_stage_sharded() builds its local table from them.
    uint64_t n_solid_local_ = 0, n_distinct_ = 0;     // from count_stage() or select_stage() to build_dictionary()
    uint32_t count_logP_ = 0;
    // the dictionary the reads are pathed against (kmer.cuh: PathDict)
    SBuf<PathSlice> path_slices;
    SBuf<uint32_t> path_bloom;
    uint32_t path_slice_words = 0;
    uint64_t n_slice_entries = 0;           // sharded: entries of the dictionary slice this rank holds
    cudaStream_t dict_stream = nullptr;     // sharded: the all-gather of the dictionary slices runs here, under the HBV stage
    cudaEvent_t dict_ready = nullptr;
    bool dict_pending = false;
    void wait_for_dictionary() { if (dict_pending) { W2R_CUDA(cudaStreamWaitEvent(c.stream, dict_ready, 0)); dict_pending = false; } }
    void build_dictionary(uint64_t n_solid_local, uint64_t n_distinct) {
        std::vector<unsigned long long> tot = {n_solid_local};
        allreduce_u64(tot, ncclSum);
        const uint64_t n_solid = tot[0];
        n_solid_local_ = n_solid_local;
        out->n_distinct = n_distinct; out->n_solid = n_solid;
        say(c, "%llu kmers counted, filtering...", (unsigned long long)n_distinct);
        say(c, "%llu / %llu kmers with Freq >= %u", (unsigned long long)n_solid, (unsigned long long)n_distinct, prm.min_freq);
        if (world > 1) return;
        EventTimer kt(c.stream);
        kt.start();
        if (n_solid > (1ull << 31) - 8) W2R_FAIL(W2RAP_ERR_OOM, "too many solid k-mers for one device's graph stage (32-bit oriented node ids); shard over more GPUs");
        const uint64_t nslots = solid_table_slots(n_solid);
        solid_slots.alloc(c, nslots);
        solid_slots.fill_ff();
        st = SolidTable{solid_slots.p, nslots};
        dense_slots.alloc(c, n_solid);
        dn = DenseNodes{st, dense_slots.p, n_solid};
        alloc_path_filter(n_solid);
        if (n_solid) W2R_TIMED(W2RAP_KT_INSERT_SOLID, W2R_LAUNCH(c, k_insert_solid, grid(n_solid, 256), 256, 0, (const ulonglong2*)cs_solid.p, n_solid, st,
                                                                   path_slice_words ? path_bloom.p : nullptr, 1u, path_slice_words, dense_slots.p));
        out->timings.dict_ms = kt.stop();
        cs_solid.release();
    }

    // ---- list ranking of the oriented nodes (unipath.cuh): splitters walk to the next splitter, the splitters alone are ranked by
    // pointer jumping, circles are cut at their minimum k-mer and ranked as paths.  On return *cur holds (tail, distance | RESOLVED)
    // of every node and *oth is scratch.  ghead (sharded runs): nodes whose predecessor lives on another rank.
    template <class V>
    void list_ranking(const V& nodes, SBuf<uint32_t>& next0, const uint8_t* ghead, uint64_t nn, SBuf<RankState>& A, SBuf<RankState>& B, RankState** cur_out, RankState** oth_out) {
        SBuf<int> flags(c, 4); flags.zero();
        SBuf<unsigned long long> scal(c, 4); scal.zero();
        // every strand head is a splitter (two per edge: up to 2 * n_solid on a graph of one-k-mer edges) plus ~1/64 of all nodes
        // by the hash rule: count them first, then size the list exactly
        W2R_LAUNCH(c, k_count_splitters, grid(nn, 256), 256, 0, next0.p, ghead, nn, scal.p + 3);
        const uint64_t nsp = d2h_scalar(c, scal.p + 3);
        SBuf<uint32_t> splist(c, nsp);
        W2R_CUDA(cudaMemsetAsync(A.p, 0xff, A.bytes(), c.stream));     // label = {NIL, ...}
        W2R_CUDA(cudaMemsetAsync(scal.p + 3, 0, 8, c.stream));
        W2R_LAUNCH(c, k_list_splitters, grid(nn, 256), 256, 0, next0.p, ghead, nn, splist.p, nsp, scal.p + 3);
        if (nsp) W2R_TIMED(W2RAP_KT_SPLITTER_WALK, W2R_LAUNCH(c, k_splitter_walk, grid(nsp, 256), 256, 0, (const uint32_t*)next0.p, (const uint32_t*)splist.p, nsp, A.p, B.p));
        unsigned long long prev_un = ~0ull;
        if (nsp) {
            for (int round = 0; round < 48; ++round) {
                W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
                W2R_LAUNCH(c, k_rank_step_inplace, grid(nsp, 256), 256, 0, (const uint32_t*)splist.p, nsp, (unsigned long long*)B.p, scal.p);
                unsigned long long un = d2h_scalar(c, scal.p);
                if (un == 0 || un == prev_un) { prev_un = un; break; }
                prev_un = un;
            }
        }
        W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
        W2R_TIMED(W2RAP_KT_SPLITTER_FINISH, W2R_LAUNCH(c, k_splitter_finish, grid(nn, 256), 256, 0, next0.p, nn, A.p, (const RankState*)B.p, scal.p));
        prev_un = d2h_scalar(c, scal.p);
        RankState* cur = A.p; RankState* oth = B.p;
        if (prev_un) {   // smooth circles (:332-335)
            uint64_t ncyc = prev_un;
            SBuf<uint32_t> list(c, ncyc);
            splist.release();
            W2R_CUDA(cudaMemsetAsync(scal.p + 1, 0, 8, c.stream));
            W2R_LAUNCH(c, k_collect_unresolved, grid(nn, 256), 256, 0, cur, nn, list.p, scal.p + 1);
            if (d2h_scalar(c, scal.p + 1) != ncyc) W2R_FAIL(W2RAP_ERR_INTERNAL, "unresolved node count changed between kernels");
            // minimum canonical k-mer per cycle by pointer doubling.  `cur` holds the final ranks of the path nodes and is
            // preserved; the cycle work ping-pongs between `oth` and D, touching only cycle entries.
            SBuf<RankState> D(c, nn);   // second buffer for cycle work (only cycle entries are touched)
            RankState* x0 = oth; RankState* x1 = D.p;
            W2R_LAUNCH(c, k_cycle_init, grid(ncyc, 256), 256, 0, list.p, ncyc, next0.p, x0);
            for (int round = 0; round < 40; ++round) {
                W2R_CUDA(cudaMemsetAsync(flags.p + 1, 0, sizeof(int), c.stream));
                W2R_LAUNCH(c, k_cycle_step, grid(ncyc, 256), 256, 0, list.p, ncyc, nodes, x0, x1, flags.p + 1);
                std::swap(x0, x1);
                if (!d2h_scalar(c, flags.p + 1)) break;
            }
            W2R_LAUNCH(c, k_cycle_cut, grid(ncyc, 256), 256, 0, list.p, ncyc, x0, next0.p);
            // the cycles are now paths: rank them
            W2R_LAUNCH(c, k_rank_init_list, grid(ncyc, 256), 256, 0, list.p, ncyc, next0.p, x0);
            for (int round = 0; round < 40; ++round) {
                W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
                W2R_LAUNCH(c, k_rank_step, grid(ncyc, 256), 256, 0, list.p, ncyc, x0, x1, scal.p);
                std::swap(x0, x1);
                unsigned long long un = d2h_scalar(c, scal.p);
                if (un == 0) break;
                if (round == 39) W2R_FAIL(W2RAP_ERR_INTERNAL, "circle ranking did not converge");
            }
            W2R_LAUNCH(c, k_copy_list, grid(ncyc, 256), 256, 0, list.p, ncyc, x0, cur);
            W2R_CUDA(cudaStreamSynchronize(c.stream));
        }
        *cur_out = cur; *oth_out = oth;
    }

    // Edge ids, lengths and byte offsets from the heads of the kept strands (E of them, in any order): deterministic edge order =
    // sorted by sequence == sorted by the first 60 bases (each oriented k-mer heads at most one edge).  edge_of[h_idx] = edge id.
    void edges_from_heads(SBuf<uint32_t>& h_idx, SBuf<uint32_t>& h_n, SBuf<uint64_t>& h_w0, SBuf<uint64_t>& h_w1, SBuf<uint32_t>& edge_of) {
        SBuf<uint32_t> perm(c, E), tmp(c, E);
        if (E) {
            W2R_LAUNCH(c, k_rs_iota, grid(E, 256), 256, 0, perm.p, (uint32_t)E);
            SortWord words[2] = {{h_w1.p, 8, 64}, {h_w0.p, 0, 64}};
            radix_sort_perm(c, perm.p, tmp.p, (uint32_t)E, words, 2);
        }
        edge_len.alloc(c, E);
        SBuf<uint32_t> nbytes(c, E);
        if (E) W2R_LAUNCH(c, k_assign_edges, grid(E, 256), 256, 0, perm.p, E, h_idx.p, h_n.p, edge_of.p, edge_len.p, nbytes.p);
        edge_off.alloc(c, E + 1);
        SBuf<unsigned long long> tot(c, 1);
        exclusive_scan<uint32_t, unsigned long long>(c, nbytes.p, E, (unsigned long long*)edge_off.p, tot.p);
        edge_bytes = E ? d2h_scalar(c, tot.p) : 0;
        W2R_CUDA(cudaMemcpyAsync(edge_off.p + E, &edge_bytes, 8, cudaMemcpyHostToDevice, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        edge_bases.alloc(c, (edge_bytes + 3 + 32) & ~3ull);
        edge_bases.zero();
    }

    // ---- buildEdges (BuildReadQGraph.cc:314-339) over the dense nodes; at the end the table slots take their nodes' results
    void unipath_stage() {
        const uint64_t nn = 2 * dn.size();
        SBuf<uint32_t> next0(c, nn);
        SBuf<int> flags(c, 4); flags.zero();
        SBuf<unsigned long long> scal(c, 4); scal.zero();
        W2R_TIMED(W2RAP_KT_LINKS, W2R_LAUNCH(c, k_links, grid(nn, 256), 256, 0, dn, next0.p, flags.p));
        if (d2h_scalar(c, flags.p)) W2R_FAIL(W2RAP_ERR_INTERNAL, "a neighbour k-mer promised by a pruned context is missing (reference: ForceAssert in EdgeBuilder::lookup)");
        // A: label, then the final (tail, distance) of every node; B: splitter states (never empty: list_ranking fills A whole)
        SBuf<RankState> A(c, std::max<uint64_t>(nn, 1)), B(c, std::max<uint64_t>(nn, 1));
        RankState* cur = nullptr; RankState* oth = nullptr;
        list_ranking(dn, next0, nullptr, nn, A, B, &cur, &oth);
        const RankState* R = cur;
        SBuf<uint8_t> keep(c, nn); keep.zero();
        W2R_LAUNCH(c, k_strand_decide, grid(nn, 256), 256, 0, dn, R, keep.p, flags.p + 2);
        if (d2h_scalar(c, flags.p + 2)) W2R_FAIL(W2RAP_ERR_EDGE_TOO_LONG, "an edge is longer than 2^24 k-mers (reference: KDef offset is 24 bits)");
        // heads of kept strands = edges.  Upper bound: one per solid k-mer.
        uint64_t cap = out->n_solid;
        SBuf<uint32_t> h_node(c, cap), h_n(c, cap);
        SBuf<uint64_t> h_w0(c, cap), h_w1(c, cap);
        W2R_CUDA(cudaMemsetAsync(scal.p + 2, 0, 8, c.stream));
        W2R_LAUNCH(c, k_collect_heads, grid(nn, 256), 256, 0, dn, R, keep.p, h_node.p, h_w0.p, h_w1.p, h_n.p, scal.p + 2, cap);
        E = d2h_scalar(c, scal.p + 2);
        if (E > cap) W2R_FAIL(W2RAP_ERR_INTERNAL, "more edges than solid k-mers");
        SBuf<uint32_t> edge_of_head(c, nn); edge_of_head.fill_ff();
        edges_from_heads(h_node, h_n, h_w0, h_w1, edge_of_head);
        W2R_TIMED(W2RAP_KT_EMIT_EDGES, W2R_LAUNCH(c, k_emit_edges, grid(nn, 256), 256, 0, dn, R, edge_of_head.p, edge_off.p, edge_bases.p));
        W2R_LAUNCH(c, k_backfill_slots, grid(st.size(), 256), 256, 0, st, (const SolidSlot*)dense_slots.p);
        dense_slots.release(); dn = DenseNodes{st, nullptr, 0};
        W2R_CUDA(cudaStreamSynchronize(c.stream));
    }

    // ---- multi-GPU plumbing of the sharded graph stage
    // all-gather of variable-size contributions (n_mine elements of T from every rank, in rank order).  off[r] = first element of
    // rank r, off[world] = total.
    template <class T>
    void allgather_v(const T* mine, uint64_t n_mine, SBuf<T>& all, std::vector<uint64_t>& off) {
        std::vector<unsigned long long> per(world, 0ull);
        per[rank] = n_mine;
        allreduce_u64(per, ncclSum);
        off.assign(world + 1, 0);
        for (int r = 0; r < world; ++r) off[r + 1] = off[r] + per[r];
        all.alloc(c, off[world] + 1);
        NcclApi& n = NcclApi::get();
        nccl_check(n.GroupStart(), "group start");
        for (int r = 0; r < world; ++r)
            if (per[r]) nccl_check(n.Broadcast(r == rank ? (const void*)mine : (const void*)(all.p + off[r]), all.p + off[r], per[r] * sizeof(T), ncclUint8, r, comm, c.stream), "broadcast");
        nccl_check(n.GroupEnd(), "group end");
        xchg_bytes += n_mine * sizeof(T) * (uint64_t)(world - 1);
    }

    // ---- recomputeAdjacencies + buildEdges (kmers/ReadPather.h:307-346, BuildReadQGraph.cc:99-339) over a dictionary that stays
    // sharded by minimiser owner (shardgraph.cuh): neighbour queries -> ghost entries, local list ranking, chain-end records
    // gathered and ranked on every rank, edge ids from a global sort, edge bases by all-reduce; finally the finished entries are
    // gathered into the pathing dictionary.  `solid` = the solid records {w0, w1 | raw ctx} this rank owns.
    void graph_stage_sharded(SBuf<ulonglong2>& solid, uint64_t n_local, uint32_t logP) {
        EventTimer xt(c.stream);
        float xms = 0;
        const uint32_t me = (uint32_t)rank, W = (uint32_t)world;
        SBuf<int> flags(c, 8); flags.zero();
        SBuf<unsigned long long> scal(c, 8); scal.zero();
        trace_mark("(before graph stage)");
        // -- round 1: neighbour queries from the solid records
        kt_.begin(W2RAP_KT_SG_QUERIES);
        uint64_t qcap = std::max<uint64_t>(1024, n_local / 4);
        SBuf<ulonglong2> qkeys;
        SBuf<unsigned long long> qcount(c, W);
        SBuf<uint64_t> qbase(c, W);
        std::vector<unsigned long long> qn(W, 0);
        for (int attempt = 0;; ++attempt) {
            if (attempt > 2) W2R_FAIL(W2RAP_ERR_INTERNAL, "neighbour query buffers did not converge");
            qkeys.alloc(c, W * qcap);
            std::vector<uint64_t> qb(W);
            for (uint32_t d = 0; d < W; ++d) qb[d] = d * qcap;
            W2R_CUDA(cudaMemcpyAsync(qbase.p, qb.data(), W * 8, cudaMemcpyHostToDevice, c.stream));
            qcount.zero();
            if (n_local) W2R_LAUNCH(c, k_neighbour_queries, grid(n_local, 256), 256, 0, solid.p, n_local, logP, W, me, QueryOut{qkeys.p, qbase.p, qcount.p, qcap});
            W2R_CUDA(cudaMemcpyAsync(qn.data(), qcount.p, W * 8, cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));
            unsigned long long mx = 0;
            for (auto v : qn) mx = std::max(mx, v);
            if (mx <= qcap) break;
            qcap = mx + mx / 32 + 64;
        }
        uint64_t nq_total = 0;
        for (auto v : qn) nq_total += v;
        kt_.end();
        trace_mark("graph: queries");
        // -- the local table: owned entries now, ghosts later
        const uint64_t nslots = solid_table_slots(n_local + nq_total);
        if (nslots > (1ull << 31) - 8) W2R_FAIL(W2RAP_ERR_OOM, "too many solid k-mers per GPU for 32-bit oriented node ids; shard over more GPUs");
        solid_slots.alloc(c, nslots);
        solid_slots.fill_ff();
        st = SolidTable{solid_slots.p, nslots};
        if (n_local) W2R_TIMED(W2RAP_KT_INSERT_SOLID, W2R_LAUNCH(c, k_insert_solid, grid(n_local, 256), 256, 0, (const ulonglong2*)solid.p, n_local, st, (uint32_t*)nullptr, 1u, 0u, (SolidSlot*)nullptr));
        solid.release();
        trace_mark("graph: local table");
        // -- keys to the owners, slots back
        kt_.begin(W2RAP_KT_SG_QUERIES);
        xt.start();
        SBuf<unsigned long long> rcount(c, W);
        alltoall_slabs(qcount.p, rcount.p, sizeof(unsigned long long));
        std::vector<unsigned long long> rn(W, 0);
        W2R_CUDA(cudaMemcpyAsync(rn.data(), rcount.p, W * 8, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        std::vector<size_t> q_off(W), q_cnt(W), r_off(W), r_cnt(W);
        uint64_t nr_total = 0;
        for (uint32_t d = 0; d < W; ++d) { q_off[d] = d * qcap; q_cnt[d] = qn[d]; r_off[d] = nr_total; r_cnt[d] = rn[d]; nr_total += rn[d]; if (d != me) xchg_bytes += qn[d] * 16 + rn[d] * 8; }
        auto scaled = [](const std::vector<size_t>& v, size_t k) { std::vector<size_t> o(v.size()); for (size_t i = 0; i < v.size(); ++i) o[i] = v[i] * k; return o; };
        SBuf<ulonglong2> rkeys(c, nr_total + 1);
        alltoall_v(qkeys.p, scaled(q_off, 16), scaled(q_cnt, 16), rkeys.p, scaled(r_off, 16), scaled(r_cnt, 16));
        SBuf<uint32_t> rreply(c, nr_total + 1), qreply(c, W * qcap), gslot(c, W * qcap);
        if (nr_total) W2R_LAUNCH(c, k_answer_queries, grid(nr_total, 256), 256, 0, st, (const ulonglong2*)rkeys.p, nr_total, rreply.p);
        alltoall_v(rreply.p, scaled(r_off, 4), scaled(r_cnt, 4), qreply.p, scaled(q_off, 4), scaled(q_cnt, 4));
        xms += xt.stop();
        rkeys.release();
        for (uint32_t d = 0; d < W; ++d)
            if (qn[d]) W2R_LAUNCH(c, k_insert_ghosts, grid(qn[d], 256), 256, 0, st, (const ulonglong2*)qkeys.p + d * qcap, (const uint32_t*)qreply.p + d * qcap, (uint64_t)qn[d], d, gslot.p + d * qcap);
        qkeys.release();
        kt_.end();
        trace_mark("graph: ghosts");
        // -- adjacency pruning of the owned entries (ghosts only answer membership); then the ghosts' pruned contexts
        W2R_TIMED(W2RAP_KT_ADJACENCY, W2R_LAUNCH(c, k_adjacency, grid(st.size(), 256), 256, 0, st));
        kt_.begin(W2RAP_KT_SG_QUERIES);
        xt.start();
        SBuf<uint32_t> rctx(c, nr_total + 1), qctx(c, W * qcap);
        if (nr_total) W2R_LAUNCH(c, k_gather_ctx, grid(nr_total, 256), 256, 0, st, (const uint32_t*)rreply.p, nr_total, rctx.p);
        alltoall_v(rctx.p, scaled(r_off, 4), scaled(r_cnt, 4), qctx.p, scaled(q_off, 4), scaled(q_cnt, 4));
        xms += xt.stop();
        for (uint32_t d = 0; d < W; ++d)
            if (qn[d]) W2R_LAUNCH(c, k_apply_ghost_ctx, grid(qn[d], 256), 256, 0, st, (const uint32_t*)gslot.p + d * qcap, (const uint32_t*)qctx.p + d * qcap, (uint64_t)qn[d]);
        kt_.end();
        rreply.release(); qreply.release(); gslot.release(); rctx.release(); qctx.release();
        trace_mark("graph: adjacency");
        // -- successor links; a node whose predecessor is a ghost heads a local piece
        const uint64_t nn = 2 * st.size();
        SBuf<uint32_t> next0(c, nn);
        SBuf<uint8_t> ghead(c, nn); ghead.zero();
        W2R_TIMED(W2RAP_KT_LINKS, W2R_LAUNCH(c, k_links_sharded, grid(nn, 256), 256, 0, st, next0.p, ghead.p, flags.p));
        if (d2h_scalar(c, flags.p)) W2R_FAIL(W2RAP_ERR_INTERNAL, "a neighbour k-mer promised by a pruned context is missing (reference: ForceAssert in EdgeBuilder::lookup)");
        SBuf<RankState> A(c, nn), B(c, nn);
        RankState* cur = nullptr; RankState* oth = nullptr;
        SBuf<PieceRec> pieces;             // all pieces of all ranks
        SBuf<uint32_t> nxt, flip;
        SBuf<RankState> S;
        uint64_t np = 0, npl_last = 0;
        uint32_t piece0 = 0;
        uint32_t* lpiece = nullptr;
        for (int iteration = 0;; ++iteration) {
            if (iteration > 1) W2R_FAIL(W2RAP_ERR_INTERNAL, "circles left after cutting them");
            list_ranking(st, next0, ghead.p, nn, A, B, &cur, &oth);
            trace_mark("graph: links+list ranking");
            // -- round 2: one record per local chain, gathered on every rank
            kt_.begin(W2RAP_KT_SG_PIECES);
            lpiece = reinterpret_cast<uint32_t*>(oth);          // scratch: local piece index per tail node ...
            uint32_t* lhead = lpiece + nn;                      // ... and per head node (the 8-byte rank array holds 2 * nn words)
            W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
            W2R_LAUNCH(c, k_count_piece_heads, grid(nn, 256), 256, 0, next0.p, (const uint8_t*)ghead.p, nn, scal.p);
            const uint64_t npl = d2h_scalar(c, scal.p);
            SBuf<PieceRec> lp(c, npl);
            W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
            W2R_LAUNCH(c, k_emit_pieces, grid(nn, 256), 256, 0, st, (const uint32_t*)next0.p, (const uint8_t*)ghead.p, (const RankState*)cur, me, lp.p, npl, scal.p, lpiece, lhead);
            if (npl) W2R_LAUNCH(c, k_piece_flips, grid(npl, 256), 256, 0, lp.p, npl, (const uint32_t*)lhead);
            xt.start();
            std::vector<uint64_t> poff;
            allgather_v(lp.p, npl, pieces, poff);
            xms += xt.stop();
            np = poff[W]; piece0 = (uint32_t)poff[me]; npl_last = npl;
            trace_mark("graph: pieces gathered");
            if (np >= (1ull << 32) - 8) W2R_FAIL(W2RAP_ERR_OOM, "more than 2^32 chain pieces");
            lp.release();
            uint64_t msz = 64;
            while (msz < 2 * np) msz <<= 1;
            SBuf<uint64_t> mkeys(c, msz); mkeys.fill_ff();
            SBuf<uint32_t> mvals(c, msz);
            GidMap gm{mkeys.p, mvals.p, msz - 1};
            nxt.alloc(c, np); flip.alloc(c, np); S.alloc(c, np);
            SBuf<uint64_t> poff_dev(c, W + 1);
            W2R_CUDA(cudaMemcpyAsync(poff_dev.p, poff.data(), (W + 1) * 8, cudaMemcpyHostToDevice, c.stream));
            if (np) {
                W2R_LAUNCH(c, k_gidmap_insert, grid(np, 256), 256, 0, (const PieceRec*)pieces.p, np, gm);
                W2R_LAUNCH(c, k_piece_link, grid(np, 256), 256, 0, (const PieceRec*)pieces.p, np, gm, (const uint64_t*)poff_dev.p, nxt.p, flip.p, flags.p + 1);
                W2R_LAUNCH(c, k_piece_rank_init, grid(np, 256), 256, 0, (const PieceRec*)pieces.p, (const uint32_t*)nxt.p, np, S.p);
            }
            if (d2h_scalar(c, flags.p + 1)) W2R_FAIL(W2RAP_ERR_INTERNAL, "a chain piece points at a node that heads no piece");
            unsigned long long un = 0, prev = ~0ull;
            for (int round = 0; round < 64 && np; ++round) {
                for (int sub = 0; sub < 3; ++sub) {           // (three doubling steps per host round trip; the count is of the last)
                    W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
                    W2R_LAUNCH(c, k_piece_rank_step, grid(np, 256), 256, 0, (unsigned long long*)S.p, np, scal.p);
                }
                un = d2h_scalar(c, scal.p);
                if (un == 0 || un == prev) break;
                prev = un;
            }
            kt_.end();
            if (un == 0) break;
            // -- circles that span ranks (BuildReadQGraph.cc:126-180): rare and small, resolved on the host.  Label every circle by
            // walking the piece links, gather the circle nodes from all ranks, cut each circle at its minimum canonical k-mer.
            std::vector<uint32_t> nxt_h(np);
            std::vector<RankState> S_h(np);
            W2R_CUDA(cudaMemcpyAsync(nxt_h.data(), nxt.p, np * 4, cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaMemcpyAsync(S_h.data(), S.p, np * 8, cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
            W2R_LAUNCH(c, k_collect_cycle_nodes, grid(nn, 256), 256, 0, st, (const uint32_t*)next0.p, (const RankState*)cur, (const uint32_t*)lpiece, piece0, (const RankState*)S.p, me,
                       (CycleNode*)nullptr, (uint64_t)0, scal.p);
            const uint64_t ncl = d2h_scalar(c, scal.p);
            SBuf<CycleNode> cyc_local(c, ncl), cyc_all;
            W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
            W2R_LAUNCH(c, k_collect_cycle_nodes, grid(nn, 256), 256, 0, st, (const uint32_t*)next0.p, (const RankState*)cur, (const uint32_t*)lpiece, piece0, (const RankState*)S.p, me,
                       cyc_local.p, ncl, scal.p);
            std::vector<uint64_t> coff;
            allgather_v(cyc_local.p, ncl, cyc_all, coff);
            std::vector<CycleNode> cn(coff[W]);
            W2R_CUDA(cudaMemcpyAsync(cn.data(), cyc_all.p, cn.size() * sizeof(CycleNode), cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));
            std::vector<uint32_t> lab(np, NIL);
            for (uint64_t i = 0; i < np; ++i) {
                if ((S_h[i].y & RANK_RESOLVED) || lab[i] != NIL) continue;
                uint32_t mn = (uint32_t)i;
                for (uint32_t j = nxt_h[i]; j != i; j = nxt_h[j]) mn = std::min(mn, j);
                lab[i] = mn;
                for (uint32_t j = nxt_h[i]; j != i; j = nxt_h[j]) lab[j] = mn;
            }
            std::sort(cn.begin(), cn.end(), [&](const CycleNode& a, const CycleNode& b) {
                const uint32_t la = lab[a.piece], lb = lab[b.piece];
                if (la != lb) return la < lb;
                if (a.w0 != b.w0) return a.w0 < b.w0;
                if (a.w1 != b.w1) return a.w1 < b.w1;
                return a.gid < b.gid;
            });
            std::vector<uint64_t> heads_g, tails_g;            // (kmin,+) becomes a head, (kmin,-) a tail
            for (size_t i = 0; i < cn.size(); ++i) {
                if (i > 0 && lab[cn[i].piece] == lab[cn[i - 1].piece]) continue;
                for (size_t j = i; j < cn.size() && lab[cn[j].piece] == lab[cn[i].piece] && cn[j].w0 == cn[i].w0 && cn[j].w1 == cn[i].w1; ++j)
                    if (cn[j].gid & 1ull) tails_g.push_back(cn[j].gid); else heads_g.push_back(cn[j].gid);
            }
            std::sort(heads_g.begin(), heads_g.end()); std::sort(tails_g.begin(), tails_g.end());
            SBuf<uint64_t> hg(c, heads_g.size() + 1), tg(c, tails_g.size() + 1);
            W2R_CUDA(cudaMemcpyAsync(hg.p, heads_g.data(), heads_g.size() * 8, cudaMemcpyHostToDevice, c.stream));
            W2R_CUDA(cudaMemcpyAsync(tg.p, tails_g.data(), tails_g.size() * 8, cudaMemcpyHostToDevice, c.stream));
            if (ncl) W2R_LAUNCH(c, k_apply_cycle_cuts, grid(ncl, 256), 256, 0, st, next0.p, ghead.p, me, (const CycleNode*)cyc_local.p, ncl, (const uint64_t*)hg.p, (uint32_t)heads_g.size(),
                                (const uint64_t*)tg.p, (uint32_t)tails_g.size());
            W2R_CUDA(cudaStreamSynchronize(c.stream));       // heads_g / tails_g leave scope
        }
        trace_mark("graph: pieces ranked");
        // -- strands: even lengths from the piece records (every rank computes them), odd lengths by the owner of the middle k-mer
        kt_.begin(W2RAP_KT_SG_EDGES);
        PieceView pv{pieces.p, flip.p, S.p, np};
        SBuf<uint8_t> is_head(c, np + 4), keepp(c, np + 4);
        SBuf<uint32_t> chain_n(c, np + 1);
        is_head.zero(); keepp.zero();
        if (np) W2R_LAUNCH(c, k_chain_tails, grid(np, 256), 256, 0, pv, (const uint32_t*)nxt.p, is_head.p, chain_n.p, keepp.p, flags.p + 2);
        SBuf<PieceInfo> pinfo(c, np + 1);
        if (np) W2R_LAUNCH(c, k_piece_info, grid(np, 256), 256, 0, pv, pinfo.p);
        if (npl_last) W2R_LAUNCH(c, k_piece_keep_odd, grid(npl_last, 256), 256, 0, st, (const uint32_t*)next0.p, (const PieceRec*)pieces.p, (const PieceInfo*)pinfo.p, piece0, npl_last, keepp.p);
        xt.start();
        if (np) nccl_check(NcclApi::get().AllReduce(keepp.p, keepp.p, np, ncclUint8, ncclMax, comm, c.stream), "all-reduce");
        xms += xt.stop();
        if (d2h_scalar(c, flags.p + 2)) W2R_FAIL(W2RAP_ERR_EDGE_TOO_LONG, "an edge is longer than 2^24 k-mers (reference: KDef offset is 24 bits)");
        trace_mark("graph: strands");
        // -- edges: kept heads sorted by k-mer (identical on every rank), emission by the owners, all-reduce of the bases
        SBuf<uint32_t> h_piece(c, np + 1), h_n(c, np + 1);
        SBuf<uint64_t> h_w0(c, np + 1), h_w1(c, np + 1);
        W2R_CUDA(cudaMemsetAsync(scal.p, 0, 8, c.stream));
        if (np) W2R_LAUNCH(c, k_collect_head_pieces, grid(np, 256), 256, 0, pv, (const uint8_t*)is_head.p, (const uint8_t*)keepp.p, (const uint32_t*)chain_n.p, h_piece.p, h_w0.p, h_w1.p, h_n.p, scal.p, np);
        E = d2h_scalar(c, scal.p);
        SBuf<uint32_t> edge_of_piece(c, np + 1); edge_of_piece.fill_ff();
        edges_from_heads(h_piece, h_n, h_w0, h_w1, edge_of_piece);
        if (np) W2R_LAUNCH(c, k_piece_edges, grid(np, 256), 256, 0, pinfo.p, np, (const uint32_t*)edge_of_piece.p);
        kt_.end();
        W2R_TIMED(W2RAP_KT_EMIT_EDGES, W2R_LAUNCH(c, k_emit_edges_sharded, grid(nn, 256), 256, 0, st, (const uint32_t*)next0.p, (const RankState*)cur, (const uint32_t*)lpiece,
                                                   (const PieceInfo*)pinfo.p + piece0, (const uint64_t*)edge_off.p, edge_bases.p));
        kt_.begin(W2RAP_KT_SG_EDGES);
        xt.start();
        const uint64_t ebw = (edge_bytes + 3) / 4;          // (disjoint bits: a sum of 32-bit words is their OR)
        if (ebw) nccl_check(NcclApi::get().AllReduce(edge_bases.p, edge_bases.p, ebw, ncclUint32, ncclSum, comm, c.stream), "all-reduce");
        xchg_bytes += ebw * 4 + np;
        kt_.end();
        kt_.begin(W2RAP_KT_SG_DICT);
        trace_mark("graph: edges");
        // -- the finished entries (pruned context, edge, offset) become the dictionary the reads are pathed against: re-sharded by
        // k-mer hash (all-to-all), slice r built on rank r in peer-mappable memory, filter slices all-gathered (kmer.cuh: PathDict)
        xms += xt.stop();
        next0.release(); ghead.release(); A.release(); B.release();
        pieces.release(); nxt.release(); flip.release(); S.release();
        uint64_t ecap = std::max<uint64_t>(1024, n_local / W + n_local / (4 * W));
        SBuf<SolidSlot> ebuck;
        SBuf<unsigned long long> ecount(c, W);
        std::vector<unsigned long long> en(W, 0);
        for (int attempt = 0;; ++attempt) {
            if (attempt > 2) W2R_FAIL(W2RAP_ERR_INTERNAL, "dictionary slice buffers did not converge");
            ebuck.alloc(c, W * ecap);
            ecount.zero();
            W2R_LAUNCH(c, k_dump_owned_sliced, grid(st.size(), 256), 256, 0, st, W, ebuck.p, ecap, ecount.p);
            W2R_CUDA(cudaMemcpyAsync(en.data(), ecount.p, W * 8, cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));
            unsigned long long mx = 0, sum = 0;
            for (auto v : en) { mx = std::max(mx, v); sum += v; }
            if (sum != n_local) W2R_FAIL(W2RAP_ERR_INTERNAL, "owned entries lost in the local table");
            if (mx <= ecap) break;
            ecap = mx + mx / 64 + 64;
        }
        solid_slots.release();
        xt.start();
        SBuf<unsigned long long> ercount(c, W);
        alltoall_slabs(ecount.p, ercount.p, sizeof(unsigned long long));
        std::vector<unsigned long long> ern(W, 0);
        W2R_CUDA(cudaMemcpyAsync(ern.data(), ercount.p, W * 8, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        std::vector<size_t> es_off(W), es_cnt(W), er_off(W), er_cnt(W);
        uint64_t n_mine = 0;
        for (uint32_t d = 0; d < W; ++d) { es_off[d] = d * ecap; es_cnt[d] = en[d]; er_off[d] = n_mine; er_cnt[d] = ern[d]; n_mine += ern[d]; if (d != me) xchg_bytes += en[d] * sizeof(SolidSlot); }
        SBuf<SolidSlot> erecv(c, n_mine + 1);
        alltoall_v(ebuck.p, scaled(es_off, sizeof(SolidSlot)), scaled(es_cnt, sizeof(SolidSlot)), erecv.p, scaled(er_off, sizeof(SolidSlot)), scaled(er_cnt, sizeof(SolidSlot)));
        xms += xt.stop();
        ebuck.release();
        kt_.end();
        // my slice, built in place inside the buffer that will hold all W slices (equal sizes: the all-gather wants them so)
        std::vector<unsigned long long> mxn = {n_mine}, tot = {n_local};
        allreduce_u64(mxn, ncclMax);
        allreduce_u64(tot, ncclSum);
        const uint64_t n_solid = tot[0];
        const uint64_t sslots = solid_table_slots(mxn[0]);            // (load 0.75 would save a fifth of the transfer, but cost the path kernel 25 %: measured)
        solid_slots.alloc(c, (size_t)W * sslots);
        SolidSlot* slice = solid_slots.p + (size_t)me * sslots;
        W2R_CUDA(cudaMemsetAsync(slice, 0xff, sslots * sizeof(SolidSlot), c.stream));
        st = SolidTable{slice, sslots};
        n_slice_entries = n_mine;
        // filter: every rank sets the bits of its own slice while it inserts; the slices are all-gathered in place
        alloc_path_filter(n_solid);
        if (n_mine) W2R_TIMED(W2RAP_KT_INSERT_SOLID, W2R_LAUNCH(c, k_insert_entries, grid(n_mine, 256), 256, 0, (const SolidSlot*)erecv.p, n_mine, st,
                                                                  path_slice_words ? path_bloom.p : nullptr, W, path_slice_words));
        erecv.release();
        kt_.begin(W2RAP_KT_SG_DICT);
        trace_mark("graph: my dictionary slice");
        // Every rank paths against ALL slices.  They are replicated with one bulk all-gather of finished table memory (large
        // contiguous NVLink transfers, no insert work on the receivers).  Tried first: leaving the slices where they were built and
        // reading them from the path kernels through peer-mapped memory (CUDA IPC) — correct, but fine-grained remote LOADS over NVLink
        // are latency-serialised: the path kernel went from 24 ms to 426 ms on two GPUs.
        // (on a side stream: the HBV vertices, which only need the edges, are computed under the transfer; path_stage() waits)
        if (!dict_stream) { W2R_CUDA(cudaStreamCreateWithFlags(&dict_stream, cudaStreamNonBlocking)); W2R_CUDA(cudaEventCreateWithFlags(&dict_ready, cudaEventDisableTiming)); }
        W2R_CUDA(cudaEventRecord(dict_ready, c.stream));
        W2R_CUDA(cudaStreamWaitEvent(dict_stream, dict_ready, 0));
        nccl_check(NcclApi::get().AllGather(slice, solid_slots.p, sslots * sizeof(SolidSlot), ncclUint8, comm, dict_stream), "all-gather");
        if (path_slice_words) nccl_check(NcclApi::get().AllGather(path_bloom.p + (size_t)me * path_slice_words, path_bloom.p, (size_t)path_slice_words * 4, ncclUint8, comm, dict_stream), "all-gather");
        W2R_CUDA(cudaEventRecord(dict_ready, dict_stream));
        dict_pending = true;
        xchg_bytes += (sslots * sizeof(SolidSlot) + (size_t)path_slice_words * 4) * (uint64_t)(W - 1);
        std::vector<PathSlice> sl(W);
        for (uint32_t r = 0; r < W; ++r) sl[r] = PathSlice{solid_slots.p + (size_t)r * sslots, sslots};
        path_slices.alloc(c, W);
        W2R_CUDA(cudaMemcpyAsync(path_slices.p, sl.data(), W * sizeof(PathSlice), cudaMemcpyHostToDevice, c.stream));
        kt_.end();
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        out->timings.graph_exchange_ms = xms;
    }

    // ---- buildHBVFromEdges (paths/long/HBVFromEdges.cc:76-154)
    void hbv_stage() {
        edge_vertices.alloc(c, 4 * E); fwd_xlat.alloc(c, E); rev_xlat.alloc(c, E);
        if (!E) { nv = nh = 0; involution.alloc(c, 0); return; }
        const uint64_t n4 = 4 * E;
        if (n4 >= (1ull << 32)) W2R_FAIL(W2RAP_ERR_OOM, "too many edges for 32-bit end indices");
        SBuf<uint64_t> kh(c, n4), k0(c, n4), k1(c, n4);
        SBuf<uint8_t> is_pal(c, E);
        W2R_LAUNCH(c, k_edge_ends, grid(n4, 128), 128, 0, edge_bases.p, edge_off.p, edge_len.p, E, kh.p, k0.p, k1.p, is_pal.p);
        SBuf<uint32_t> perm(c, n4), tmp(c, n4);
        W2R_LAUNCH(c, k_rs_iota, grid(n4, 256), 256, 0, perm.p, (uint32_t)n4);
        // EdgeEnd order = (64-bit hash, bases).  Distinct (K-1)-mers sharing a hash are a ~n^2/2^65 event, so the 8 digit passes over
        // the hash word nearly always ARE the order (ends with equal keys may come in any order: they get the same vertex); a check
        // of neighbours proves it, and if it ever fails the 23-pass sort over all three words runs instead.
        SortWord words[3] = {{k1.p, 10, 64}, {k0.p, 0, 64}, {kh.p, 0, 64}};
        static const bool full_sort = getenv("W2RAP_HBV_FULL_SORT") != nullptr;       // (test hook: keeps the long path exercised)
        SBuf<unsigned long long> coll(c, 1); coll.zero();
        if (!full_sort) {
            radix_sort_perm(c, perm.p, tmp.p, (uint32_t)n4, words + 2, 1);
            W2R_LAUNCH(c, k_hash_order_check, grid(n4, 256), 256, 0, (const uint32_t*)perm.p, n4, (const uint64_t*)kh.p, (const uint64_t*)k0.p, (const uint64_t*)k1.p, coll.p);
        }
        if (full_sort || d2h_scalar(c, coll.p)) {
            W2R_LAUNCH(c, k_rs_iota, grid(n4, 256), 256, 0, perm.p, (uint32_t)n4);
            radix_sort_perm(c, perm.p, tmp.p, (uint32_t)n4, words, 3);
        }
        SBuf<uint32_t> flag(c, n4), excl(c, n4), tot(c, 1);
        W2R_LAUNCH(c, k_vertex_flags, grid(n4, 256), 256, 0, perm.p, n4, kh.p, k0.p, k1.p, flag.p);
        exclusive_scan<uint32_t, uint32_t>(c, flag.p, n4, excl.p, tot.p);
        nv = d2h_scalar(c, tot.p);
        W2R_LAUNCH(c, k_scatter_vids, grid(n4, 256), 256, 0, perm.p, n4, flag.p, excl.p, kh.p, k0.p, k1.p, edge_vertices.p);
        SBuf<uint32_t> width(c, E), xl(c, E);
        W2R_LAUNCH(c, k_pal_widths, grid(E, 256), 256, 0, is_pal.p, E, width.p);
        exclusive_scan<uint32_t, uint32_t>(c, width.p, E, xl.p, tot.p);
        nh = d2h_scalar(c, tot.p);
        hcanon.alloc(c, nh); hleft.alloc(c, nh); hright.alloc(c, nh); involution.alloc(c, nh);
        W2R_LAUNCH(c, k_hbv_edges, grid(E, 256), 256, 0, E, is_pal.p, xl.p, edge_vertices.p, fwd_xlat.p, rev_xlat.p, hcanon.p, hleft.p, hright.p, involution.p);
        from_e.alloc(c, 4 * nv); to_e.alloc(c, 4 * nv); from_n.alloc(c, nv); to_n.alloc(c, nv);
        SBuf<uint32_t> fc(c, nv), tc(c, nv); fc.zero(); tc.zero();
        SBuf<int> bad(c, 1); bad.zero();
        W2R_LAUNCH(c, k_adj_fill, grid(nh, 256), 256, 0, nh, hleft.p, hright.p, from_e.p, to_e.p, fc.p, tc.p, bad.p);
        if (d2h_scalar(c, bad.p)) W2R_FAIL(W2RAP_ERR_INTERNAL, "a vertex has more than four edges on one side");
        W2R_LAUNCH(c, k_adj_sort, grid(nv, 128), 128, 0, nv, hleft.p, hright.p, from_e.p, to_e.p, fc.p, tc.p, from_n.p, to_n.p);
        W2R_CUDA(cudaStreamSynchronize(c.stream));
    }

    // ---- path_reads_OMP (+FixPaths)  (BuildReadQGraph.cc:829-929; large/GapToyTools.cc:322-335)
    void path_stage(SBuf<int32_t>& d_offset, SBuf<uint64_t>& d_path_off, SBuf<int32_t>& d_path_edges, uint64_t* n_path_edges, unsigned long long* pathed,
                    unsigned long long* multipathed) {
        const uint64_t n = dr.n;
        d_offset.alloc(c, n); d_path_off.alloc(c, n + 1);
        *n_path_edges = 0; *pathed = 0; *multipathed = 0;
        if (!n) { W2R_CUDA(cudaMemsetAsync(d_path_off.p, 0, 8, c.stream)); return; }
        // the dictionary the reads are pathed against (kmer.cuh: PathDict).  One GPU: the graph stage's own table as the only slice and
        // a filter built here; sharded: graph_stage_sharded() left this rank's slice, the peer-mapped slices of the others and the
        // all-gathered filter.  (The filter is not pinned in L2: its misses are sectors of a 192 MB array either way, and the
        // persisting carve-out made no difference once the kernel stopped spilling: 96 / 192 / 384 MB all 47 ms at config 2.)
        wait_for_dictionary();
        if (world == 1) {
            const PathSlice one{st.slots, st.nslots};
            path_slices.alloc(c, 1);
            W2R_CUDA(cudaMemcpyAsync(path_slices.p, &one, sizeof one, cudaMemcpyHostToDevice, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));       // (`one` leaves scope)
        }
        const PathDict dict{path_slices.p, (uint32_t)world, path_slice_words ? path_bloom.p : nullptr, path_slice_words};
        GraphView g{dict, edge_bases.p, edge_off.p, edge_len.p, fwd_xlat.p, rev_xlat.p, hcanon.p, hleft.p, hright.p, from_e.p, to_e.p, from_n.p, to_n.p};
        const ReadsView rv = dr.view();
        const unsigned block = 128;
        const uint32_t cap = 24, left_cap = 8;
        SBuf<int32_t> stage(c, n * cap), row_off(c, n);
        SBuf<PathMeta> meta(c, n);
        SBuf<uint32_t> lens(c, n);
        SBuf<unsigned long long> counters(c, 4); counters.zero();
        // resident CTAs per SM the compiler must allow for (register cap): the kernel waits on dependent DRAM fetches, so warps in flight matter
        // measured (config 2, path stage): 8 CTAs/SM (64 registers) 96 ms, 10: 105 ms, 12 (40 registers, more spills) 81.5 ms, 14/16: 86 ms
        // round 2 (walker state in shared memory, ~350 B less stack): 12 CTAs/SM 71.8 ms, 10: 59.8 ms, 8 (64 registers): 54.9 ms
        W2R_TIMED(W2RAP_KT_PATH_READS, W2R_LAUNCH(c, k_path_reads, grid(n, block, PATH_CTAS_PER_SM), block, 0, rv, g, nullptr, n, stage.p, cap, left_cap, row_off.p, meta.p, prm.apply_fixpaths));
        W2R_LAUNCH(c, k_path_lens, grid(n, 256), 256, 0, meta.p, (const uint32_t*)nullptr, n, lens.p, counters.p);
        unsigned long long cnt[3];
        W2R_CUDA(cudaMemcpyAsync(cnt, counters.p, 24, cudaMemcpyDeviceToHost, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        // rows that overflowed the small staging row are pathed again with a row that always suffices
        uint64_t n_ovf = cnt[2];
        SBuf<uint32_t> olist(c, n_ovf);
        const uint32_t cap2 = 3 * dr.max_len + 32, left2 = dr.max_len + 16;
        SBuf<int32_t> stage2(c, n_ovf * cap2), row_off2(c, n_ovf);
        SBuf<PathMeta> meta2(c, n_ovf);
        if (n_ovf) {
            W2R_CUDA(cudaMemsetAsync(counters.p + 3, 0, 8, c.stream));
            W2R_LAUNCH(c, k_collect_overflow, grid(n, 256), 256, 0, meta.p, n, olist.p, counters.p + 3);
            W2R_TIMED(W2RAP_KT_PATH_READS, W2R_LAUNCH(c, k_path_reads, grid(n_ovf, block, PATH_CTAS_PER_SM), block, 0, rv, g, (const uint32_t*)olist.p, n_ovf, stage2.p, cap2, left2,
                                                      row_off2.p, meta2.p, prm.apply_fixpaths));
            W2R_CUDA(cudaMemsetAsync(counters.p + 2, 0, 8, c.stream));
            W2R_LAUNCH(c, k_path_lens, grid(n_ovf, 256), 256, 0, meta2.p, (const uint32_t*)olist.p, n_ovf, lens.p, counters.p);
            W2R_CUDA(cudaMemcpyAsync(cnt, counters.p, 24, cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));
            if (cnt[2]) W2R_FAIL(W2RAP_ERR_INTERNAL, "a read path overflowed the worst-case staging row");
        }
        *pathed = cnt[0]; *multipathed = cnt[1];
        SBuf<unsigned long long> tot(c, 1);
        exclusive_scan<uint32_t, unsigned long long>(c, lens.p, n, (unsigned long long*)d_path_off.p, tot.p);
        *n_path_edges = d2h_scalar(c, tot.p);
        W2R_CUDA(cudaMemcpyAsync(d_path_off.p + n, n_path_edges, 8, cudaMemcpyHostToDevice, c.stream));
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        d_path_edges.alloc(c, *n_path_edges);
        W2R_LAUNCH(c, k_path_gather, grid(n, 256), 256, 0, stage.p, cap, meta.p, (const uint32_t*)nullptr, row_off.p, d_path_off.p, n, d_path_edges.p, d_offset.p);
        if (n_ovf) W2R_LAUNCH(c, k_path_gather, grid(n_ovf, 256), 256, 0, stage2.p, cap2, meta2.p, (const uint32_t*)olist.p, row_off2.p, d_path_off.p, n_ovf, d_path_edges.p, d_offset.p);
        W2R_CUDA(cudaStreamSynchronize(c.stream));
    }

    // ---- step-3 input: RepathInMemory's places (paths/long/large/Repath.cc:46-72; kernels and rules in places.cuh)
    struct PlaceSet { SBuf<uint64_t> off; SBuf<int32_t> edges; uint64_t n = 0, n_edges = 0; };
    // `in` without its duplicates, in std::vector<int> order if `sorted` (else in hash order)
    void unique_places(PlaceSet& in, PlaceSet& res, bool sorted) {
        const uint64_t M = in.n;
        res.n = res.n_edges = 0;
        if (M == 0) { res.off.alloc(c, 1); res.off.zero(); res.edges.alloc(c, 1); return; }
        if (M >= (1ull << 32) - 8) W2R_FAIL(W2RAP_ERR_OOM, "more than 2^32 places");
        PlacesView s{in.off.p, in.edges.p, M};
        SBuf<uint64_t> h(c, M);
        SBuf<uint32_t> perm(c, M), tmp(c, M), first(c, M), excl(c, M), tot(c, 1);
        SBuf<unsigned long long> coll(c, 1);
        for (int attempt = 0;; ++attempt) {
            W2R_LAUNCH(c, k_place_hash, grid(M, 256), 256, 0, s, 0x1234567ull + 0x9e3779b97f4a7c15ull * (uint64_t)attempt, h.p);
            W2R_LAUNCH(c, k_rs_iota, grid(M, 256), 256, 0, perm.p, (uint32_t)M);
            SortWord w{h.p, 0, 64};
            radix_sort_perm(c, perm.p, tmp.p, (uint32_t)M, &w, 1);
            coll.zero();
            W2R_LAUNCH(c, k_place_first, grid(M, 256), 256, 0, s, (const uint32_t*)perm.p, (const uint64_t*)h.p, first.p, coll.p);
            if (!d2h_scalar(c, coll.p)) break;                 // no two different places share a hash: equal places are neighbours
            if (attempt == 3) W2R_FAIL(W2RAP_ERR_INTERNAL, "place hashes collide under four salts");
        }
        exclusive_scan<uint32_t, uint32_t>(c, first.p, M, excl.p, tot.p);
        const uint64_t U = d2h_scalar(c, tot.p);
        SBuf<uint32_t> rep(c, U), order;
        SBuf<unsigned int> maxlen(c, 1); maxlen.zero();
        W2R_LAUNCH(c, k_place_select, grid(M, 256), 256, 0, s, (const uint32_t*)perm.p, (const uint32_t*)first.p, (const uint32_t*)excl.p, rep.p, maxlen.p);
        if (sorted && U > 1) {
            const uint32_t ml = d2h_scalar(c, maxlen.p);
            order.alloc(c, U);
            SBuf<uint32_t> tmp2(c, U);
            SBuf<uint64_t> key(c, U);
            W2R_LAUNCH(c, k_rs_iota, grid(U, 256), 256, 0, order.p, (uint32_t)U);
            int bits = 1;
            while ((1ull << bits) < nh + 2) ++bits;            // keys are hbv id + 1 (0 = the vector has ended)
            for (uint32_t pos = ml; pos-- > 0;) {              // stable LSD: last element position first
                W2R_LAUNCH(c, k_place_key, grid(U, 256), 256, 0, s, (const uint32_t*)rep.p, U, pos, key.p);
                SortWord w{key.p, 0, bits};
                radix_sort_perm(c, order.p, tmp2.p, (uint32_t)U, &w, 1);
            }
        }
        SBuf<uint32_t> olen(c, U);
        SBuf<uint64_t> tote(c, 1);
        W2R_LAUNCH(c, k_place_out_len, grid(U, 256), 256, 0, s, (const uint32_t*)rep.p, (const uint32_t*)order.p, U, olen.p);
        res.off.alloc(c, U + 1);
        exclusive_scan<uint32_t, uint64_t>(c, olen.p, U, res.off.p, tote.p);
        W2R_CUDA(cudaMemcpyAsync(res.off.p + U, tote.p, 8, cudaMemcpyDeviceToDevice, c.stream));
        const uint64_t ne = d2h_scalar(c, tote.p);
        res.edges.alloc(c, ne + 1);
        W2R_LAUNCH(c, k_place_gather, grid(U, 256), 256, 0, s, (const uint32_t*)rep.p, (const uint32_t*)order.p, U, (const uint64_t*)res.off.p, res.edges.p);
        res.n = U; res.n_edges = ne;
    }
    void places_stage(SBuf<uint64_t>& d_path_off, SBuf<int32_t>& d_path_edges) {
        const uint64_t n = dr.n;
        PlaceSet local, uniq;
        {
            PathsView pv{d_path_off.p, d_path_edges.p, n};
            SBuf<uint32_t> plen(c, n + 1), kept(c, n + 1), pidx(c, n + 1), totk(c, 1);
            SBuf<uint8_t> flip(c, n + 1);
            SBuf<uint64_t> poff(c, n + 1), tote(c, 1);
            if (n) W2R_LAUNCH(c, k_place_measure, grid(n, 256), 256, 0, pv, (const uint32_t*)hcanon.p, (const uint32_t*)edge_len.p, (const int32_t*)involution.p, prm.places_K2, plen.p, kept.p, flip.p);
            exclusive_scan<uint32_t, uint32_t>(c, kept.p, n, pidx.p, totk.p);
            exclusive_scan<uint32_t, uint64_t>(c, plen.p, n, poff.p, tote.p);
            local.n = d2h_scalar(c, totk.p);
            local.n_edges = d2h_scalar(c, tote.p);
            local.off.alloc(c, local.n + 1); local.edges.alloc(c, local.n_edges + 1);
            if (n) W2R_LAUNCH(c, k_place_fill, grid(n, 256), 256, 0, pv, (const int32_t*)involution.p, (const uint32_t*)plen.p, (const uint8_t*)flip.p, (const uint32_t*)pidx.p,
                              (const uint64_t*)poff.p, local.off.p, local.edges.p);
            W2R_CUDA(cudaMemcpyAsync(local.off.p + local.n, tote.p, 8, cudaMemcpyDeviceToDevice, c.stream));
        }
        std::vector<unsigned long long> kt = {local.n};
        allreduce_u64(kt, ncclSum);
        out->n_places_kept = kt[0];
        if (world == 1) {
            unique_places(local, uniq, true);
        } else {                                               // every rank removes its own duplicates, the rest is merged on all ranks
            PlaceSet mine, merged;
            unique_places(local, mine, false);
            local.off.release(); local.edges.release();
            SBuf<uint32_t> mylen(c, mine.n + 1), all_len;
            SBuf<uint64_t> tot(c, 1);
            if (mine.n) W2R_LAUNCH(c, k_place_lens, grid(mine.n, 256), 256, 0, (const uint64_t*)mine.off.p, mine.n, mylen.p);
            std::vector<uint64_t> loff, eoff;
            allgather_v(mylen.p, mine.n, all_len, loff);
            allgather_v(mine.edges.p, mine.n_edges, merged.edges, eoff);
            merged.n = loff[world]; merged.n_edges = eoff[world];
            merged.off.alloc(c, merged.n + 1);
            exclusive_scan<uint32_t, uint64_t>(c, all_len.p, merged.n, merged.off.p, tot.p);
            W2R_CUDA(cudaMemcpyAsync(merged.off.p + merged.n, tot.p, 8, cudaMemcpyDeviceToDevice, c.stream));
            unique_places(merged, uniq, true);
        }
        out->n_places = uniq.n; out->n_place_edges = uniq.n_edges;
        if (!(world > 1 && prm.graph_on_root_only && rank != 0)) {
            out->place_off = to_host<uint64_t>(uniq.off.p, uniq.n + 1);
            out->place_edges = to_host<int32_t>(uniq.edges.p, uniq.n_edges);
        }
        W2R_CUDA(cudaStreamSynchronize(c.stream));             // (the sets leave scope)
    }

    template <class T>
    T* to_host(const T* dptr, size_t n, cudaStream_t s = nullptr) {
        T* h = out_alloc<T>(owner, n);
        if (!n) return h;
        if (s && ((uintptr_t)h & 15) == 0 && ((uintptr_t)dptr & 15) == 0) {      // side stream: by stores, leaving the copy engine to the main stream
            k_copy_to_host<<<32, 512, 0, s>>>((const uint8_t*)dptr, (uint8_t*)h, n * sizeof(T));
            W2R_CUDA(cudaGetLastError());
            c.launches++;
        } else {
            W2R_CUDA(cudaMemcpyAsync(h, dptr, n * sizeof(T), cudaMemcpyDeviceToHost, s ? s : c.stream));
        }
        return h;
    }
    cudaStream_t copy_stream = nullptr;     // the graph travels to the host while the reads are pathed

    void begin() {
        W2R_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        g_alloc_host_ms = 0;
        kt_.s = c.stream;
        c.verbose = prm.verbose != 0;
        out->n_reads = dr.n; out->n_bases = dr.n_bases;
    }

    void run() {
        begin();
        StageTimer total(c), st_t(c);
        total.start();
        st_t.start();
        if (from_counts) {
            say(c, "selecting kmers with Freq >= %u from the counts kept at Freq >= %u", prm.min_freq, from_counts->f0);
            select_stage();
        } else {
            say(c, "creating kmers from reads...");
            count_stage();
        }
        build_dictionary(n_solid_local_, n_distinct_);
        out->timings.count_ms = st_t.stop();
        good.release();
        if (world > 1) {
            say(c, "updating adjacencies, finding edges (unique paths): dictionary sharded over %d GPUs", world);
            st_t.start(); graph_stage_sharded(cs_solid, n_solid_local_, count_logP_); out->timings.unipath_ms = st_t.stop();
        } else {
            say(c, "updating adjacencies");
            st_t.start();
            W2R_TIMED(W2RAP_KT_ADJACENCY, W2R_LAUNCH(c, k_adjacency_dense, grid(dn.size(), 256), 256, 0, dn));
            out->timings.adjacency_ms = st_t.stop();
            say(c, "finding edges (unique paths)");
            st_t.start(); unipath_stage(); out->timings.unipath_ms = st_t.stop();
        }
        say(c, "building graph...");
        st_t.start(); hbv_stage(); out->timings.hbv_ms = st_t.stop();
        // ---- the graph is final: its arrays go to the host on a second stream, under the pathing kernels
        out->n_edges = E; out->n_vertices = nv; out->n_hbv_edges = nh;
        W2R_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));     // (hbv_stage ended with a drained stream: st_t.stop())
        out->edge_len = to_host<uint32_t>(edge_len.p, E, copy_stream);
        if (!(world > 1 && prm.graph_on_root_only && rank != 0)) {
            out->edge_off = to_host<uint64_t>(edge_off.p, E + 1, copy_stream);
            out->edge_bases = to_host<uint8_t>(edge_bases.p, edge_bytes, copy_stream);
            out->edge_vertices = to_host<int32_t>(edge_vertices.p, 4 * E, copy_stream);
            out->fwd_xlat = to_host<int32_t>(fwd_xlat.p, E, copy_stream);
            out->rev_xlat = to_host<int32_t>(rev_xlat.p, E, copy_stream);
            out->involution = to_host<int32_t>(involution.p, nh, copy_stream);
        }
        SBuf<int32_t> d_offset, d_path_edges; SBuf<uint64_t> d_path_off;
        uint64_t npe = 0; unsigned long long pathed = 0, multi = 0;
        if (prm.want_paths) {
            say(c, "pathing reads into graph...");
            st_t.start(); path_stage(d_offset, d_path_off, d_path_edges, &npe, &pathed, &multi); out->timings.path_ms = st_t.stop();
            say(c, "%llu / %llu reads pathed, %llu spanning junctions", pathed, (unsigned long long)dr.n, multi);
        }
        if (prm.places_K2) {
            say(c, "constructing places from %llu paths", (unsigned long long)dr.n);
            st_t.start(); places_stage(d_path_off, d_path_edges); out->timings.places_ms = st_t.stop();
            say(c, "sorting %llu places", (unsigned long long)out->n_places_kept);
            say(c, "%llu unique places", (unsigned long long)out->n_places);
        }
        // ---- results to the host
        st_t.start();
        SBuf<unsigned long long> dig(c, 2); dig.zero();
        {   // digest of the graph: every array at its own salt
            struct Part { const void* p; size_t bytes; } parts[] = {{edge_len.p, E * 4}, {edge_bases.p, edge_bytes}, {edge_vertices.p, 4 * E * 4}, {fwd_xlat.p, E * 4}, {rev_xlat.p, E * 4}};
            uint64_t salt = 1;
            for (const Part& pt : parts) { if (pt.bytes) W2R_LAUNCH(c, k_digest_words, grid((pt.bytes + 3) / 4, 256, 4), 256, 0, (const uint8_t*)pt.p, pt.bytes, salt << 40, dig.p); ++salt; }
            if (prm.want_paths && dr.n) W2R_LAUNCH(c, k_digest_paths, grid(dr.n, 256, 8), 256, 0, dr.view(), d_offset.p, d_path_off.p, d_path_edges.p, dig.p + 1);
        }
        unsigned long long dig_h[2] = {0, 0};
        W2R_CUDA(cudaMemcpyAsync(dig_h, dig.p, 16, cudaMemcpyDeviceToHost, c.stream));
        if (prm.want_paths) {
            out->n_paths = dr.n; out->n_path_edges = npe; out->n_pathed = pathed; out->n_multipathed = multi;
            out->path_offset = to_host<int32_t>(d_offset.p, dr.n);
            out->path_off = to_host<uint64_t>(d_path_off.p, dr.n + 1);
            out->path_edges = to_host<int32_t>(d_path_edges.p, npe);
        }
        wait_for_dictionary();
        if (prm.dump_kmers == 1 && out->n_solid) {
            // (sharded: every rank dumps the dictionary slice it holds; the test hook gathers them so that every rank reports the whole)
            const uint64_t n_mine = world > 1 ? n_slice_entries : out->n_solid;
            SBuf<DumpRec> dd(c, n_mine + 1), dd_all;
            SBuf<unsigned long long> cur(c, 1); cur.zero();
            W2R_LAUNCH(c, k_dump_solid, grid(st.size(), 256), 256, 0, st, dd.p, cur.p);
            const DumpRec* src = dd.p;
            if (world > 1) { std::vector<uint64_t> doff; allgather_v(dd.p, n_mine, dd_all, doff); src = dd_all.p; }
            dump_host.resize(out->n_solid);
            W2R_CUDA(cudaMemcpyAsync(dump_host.data(), src, out->n_solid * sizeof(DumpRec), cudaMemcpyDeviceToHost, c.stream));
            W2R_CUDA(cudaStreamSynchronize(c.stream));
        }
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        W2R_CUDA(cudaStreamSynchronize(copy_stream));
        out->timings.d2h_ms = st_t.stop();
        if (E == 0 && out->edge_off) out->edge_off[0] = 0;
        uint64_t neb = 0;
        for (uint64_t i = 0; i < E; ++i) neb += out->edge_len[i];
        out->n_edge_bases = neb;
        if (prm.dump_kmers && !dump_host.empty()) {
            std::sort(dump_host.begin(), dump_host.end(), [](const DumpRec& a, const DumpRec& b) { return a.w0 < b.w0 || (a.w0 == b.w0 && a.w1 < b.w1); });
            out->n_dump = dump_host.size();
            out->dump = out_alloc<w2rap_kmer_rec>(owner, dump_host.size());
            static_assert(sizeof(DumpRec) == sizeof(w2rap_kmer_rec), "dump record layout");
            memcpy(out->dump, dump_host.data(), dump_host.size() * sizeof(DumpRec));
        }
        {   // digests (the histogram is folded in on the host: 101 words)
            uint64_t hd = 0;
            for (int i = 0; i <= 100; ++i) { uint64_t x = out->hist[i] + 0x9e3779b97f4a7c15ull * (uint64_t)(i + 1); x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; hd += x; }
            out->digest_graph = dig_h[0] + hd;
            std::vector<unsigned long long> dp = {dig_h[1]};
            allreduce_u64(dp, ncclSum);           // paths: summed over the shards
            out->digest_paths = dp[0];
        }
        out->timings.total_ms = total.stop();
        kt_.resolve(out->timings.kernel_ms);
        out->timings.alloc_host_ms = (float)g_alloc_host_ms;
        out->timings.exchange_bytes = xchg_bytes;
        out->timings.count_exchange_bytes = xchg_count_bytes;
        out->timings.n_records = n_records;
        out->timings.kernel_launches = c.launches;
        out->timings.count_launches = c.count_launches;
        say(c, "%llu edges of total length %llu; %llu vertices", (unsigned long long)E, (unsigned long long)neb, (unsigned long long)nv);
    }

    // w2rap_step2_count: the count stage alone, with the reduce keeping every k-mer seen >= f0 = prm.min_freq times and its count.
    // The kept records and counts leave the (per-call) device slab for allocations the handle owns: 17 bytes per kept k-mer.
    void run_count(w2rap_counts* h) {
        begin();
        keep_counts = true;
        StageTimer total(c);
        total.start();
        say(c, "creating kmers from reads...");
        count_stage();
        const uint64_t n = n_solid_local_;
        std::vector<unsigned long long> kept = {n};
        allreduce_u64(kept, ncclSum);              // sharded: the summary counts what all ranks keep
        out->n_distinct = n_distinct_; out->n_solid = kept[0];
        say(c, "%llu kmers counted, %llu with Freq >= %u kept", (unsigned long long)n_distinct_, kept[0], prm.min_freq);
        const double t0 = now_ms();
        cudaError_t e = cudaMallocAsync((void**)&h->solid, std::max<uint64_t>(n, 1) * sizeof(ulonglong2), c.stream);
        if (e == cudaSuccess) e = cudaMallocAsync((void**)&h->count, std::max<uint64_t>(n, 1), c.stream);
        g_alloc_host_ms += now_ms() - t0;
        W2R_CUDA(e);
        if (n) {
            W2R_CUDA(cudaMemcpyAsync(h->solid, cs_solid.p, n * sizeof(ulonglong2), cudaMemcpyDeviceToDevice, c.stream));
            W2R_CUDA(cudaMemcpyAsync(h->count, cs_count.p, n, cudaMemcpyDeviceToDevice, c.stream));
        }
        W2R_CUDA(cudaStreamSynchronize(c.stream));
        cs_solid.release(); cs_count.release(); good.release();
        h->n_kept = n; h->n_distinct = n_distinct_; h->n_kmer_instances = out->n_kmer_instances; h->logP = count_logP_;
        for (int i = 0; i <= 100; ++i) h->hist[i] = out->hist[i];
        if (!dump_host.empty()) {
            std::sort(dump_host.begin(), dump_host.end(), [](const DumpRec& a, const DumpRec& b) { return a.w0 < b.w0 || (a.w0 == b.w0 && a.w1 < b.w1); });
            out->n_dump = dump_host.size();
            out->dump = out_alloc<w2rap_kmer_rec>(owner, dump_host.size());
            memcpy(out->dump, dump_host.data(), dump_host.size() * sizeof(DumpRec));
        }
        out->timings.count_ms = out->timings.total_ms = total.stop();
        kt_.resolve(out->timings.kernel_ms);
        out->timings.alloc_host_ms = (float)g_alloc_host_ms;
        out->timings.n_records = n_records;
        out->timings.kernel_launches = c.launches;
        out->timings.count_launches = c.count_launches;
    }

    ~Pipeline() {
        // free stream-ordered buffers before the stream goes away (and not under a transfer that still writes into them)
        if (dict_stream) cudaStreamSynchronize(dict_stream);
        if (copy_stream) { cudaStreamSynchronize(copy_stream); cudaStreamDestroy(copy_stream); }
        good.release(); solid_slots.release(); dense_slots.release(); edge_bases.release(); edge_off.release(); edge_len.release();
        edge_vertices.release(); fwd_xlat.release(); rev_xlat.release(); involution.release(); hleft.release();
        cs_scal.release(); cs_flags.release(); cs_hist.release(); cs_region.release(); cs_dump.release(); cs_solid.release(); cs_count.release();
        path_slices.release(); path_bloom.release(); hright.release(); from_e.release(); to_e.release();
        hcanon.release(); from_n.release(); to_n.release();
        if (dict_stream) { cudaStreamSynchronize(dict_stream); cudaStreamDestroy(dict_stream); cudaEventDestroy(dict_ready); }
        if (c.stream) { cudaStreamSynchronize(c.stream); cudaStreamDestroy(c.stream); }
    }
};

static void validate_reads(const w2rap_reads* in) {
    if (!in) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null read store");
    if (in->n_reads && (!in->bases || !in->base_off || !in->len || !in->quals || !in->qual_off)) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null pointer in read store");
    if (in->n_reads >= (1ull << 32)) W2R_FAIL(W2RAP_ERR_BAD_ARG, "more than 2^32-1 reads on one device");
}

// Device buffers for the read stores of the host-buffer entry points.  They are kept between calls (grow-only, one set per
// device): taking them from the stream-ordered pool instead fragments it, and the 80+ GB record pool of the counting stage then
// has to be re-created by the driver on every call (measured: +120 ms per step).
struct UploadArena {
    std::mutex mu;
    bool in_use = false;
    void* buf[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t cap[5] = {0, 0, 0, 0, 0};
    static UploadArena& get(int device) { static UploadArena* a = new UploadArena[16]; return a[device & 15]; }
};
void arena_release(int device) { UploadArena& a = UploadArena::get(device); std::lock_guard<std::mutex> g(a.mu); a.in_use = false; }
static void dev_alloc(DeviceReads* d, void** p, size_t bytes, cudaStream_t s, int which) {
    if (d->arena) {
        UploadArena& a = UploadArena::get(d->device);
        if (a.cap[which] < bytes) {
            if (a.buf[which]) cudaFree(a.buf[which]);
            a.buf[which] = nullptr; a.cap[which] = 0;
            size_t want = bytes + bytes / 16;
            W2R_CUDA(cudaMalloc(&a.buf[which], want));
            a.cap[which] = want;
        }
        *p = a.buf[which];
        return;
    }
    if (d->pooled) W2R_CUDA(cudaMallocAsync(p, bytes, s)); else W2R_CUDA(cudaMalloc(p, bytes));
}
// W2RAP_UPLOAD_BATCHES=n (test hook): the host-buffer entry points split every non-empty read set into exactly n read batches, so
// that the multi-run count (one record run per batch in every partition) can be checked on small read sets.  0 when unset, -1
// when set to anything but 1..SMEM_MAX_BATCH.
static int upload_batches_override() {
    static const int n = [] {
        const char* v = getenv("W2RAP_UPLOAD_BATCHES");
        if (!v) return 0;
        char* end = nullptr;
        const long x = strtol(v, &end, 10);
        return (end != v && *end == '\0' && x >= 1 && x <= (long)SMEM_MAX_BATCH) ? (int)x : -1;
    }();
    return n;
}

// Validates the flattened store and starts its transfer.  With `batched`, the copy is issued as read batches (8 from 2^20 reads on,
// else 1, or as W2RAP_UPLOAD_BATCHES says) with an event each and NOT waited for: the pipeline consumes batch b while batch b+1 is
// in flight.  Host buffers must stay valid until the stream has drained (the entry points synchronise before returning).
static void upload(const w2rap_reads* in, int device, DeviceReads* d, cudaStream_t s, bool batched) {
    const int forced_batches = batched ? upload_batches_override() : 0;
    if (forced_batches < 0) W2R_FAIL(W2RAP_ERR_BAD_ARG, "W2RAP_UPLOAD_BATCHES must be an integer in 1..%u (the most record runs per partition the count handles)", SMEM_MAX_BATCH);
    d->device = device;
    d->n = in->n_reads;
    const uint64_t n = d->n;
    d->bases_bytes = n ? in->base_off[n] : 0;
    d->quals_bytes = n ? in->qual_off[n] : 0;
    const double t0 = now_ms();
    {   // one pass over the offsets/lengths, on a few host threads
        const unsigned nt = n > (1u << 20) ? 8u : 1u;
        std::vector<uint64_t> t_nb(nt, 0), t_inst(nt, 0), t_bad(nt, ~0ull), t_kr(nt, 0);
        std::vector<uint32_t> t_mx(nt, 0), t_kind(nt, 0);
        auto work = [&](unsigned t) {
            uint64_t lo = n * t / nt, hi = n * (t + 1) / nt, nb = 0, inst = 0, kr = 0; uint32_t mx = 0;
            for (uint64_t i = lo; i < hi; ++i) {
                uint32_t L = in->len[i];
                nb += L; if (L > mx) mx = L;
                if (L > 59) { inst += L - 59; ++kr; }
                if (in->base_off[i + 1] < in->base_off[i] || in->base_off[i + 1] - in->base_off[i] < (uint64_t)(L + 3) / 4) { t_bad[t] = i; t_kind[t] = 1; break; }
                if (in->qual_off[i + 1] <= in->qual_off[i]) { t_bad[t] = i; t_kind[t] = 2; break; }
            }
            t_nb[t] = nb; t_inst[t] = inst; t_mx[t] = mx; t_kr[t] = kr;
        };
        std::vector<std::thread> th;
        for (unsigned t = 1; t < nt; ++t) th.emplace_back(work, t);
        work(0);
        for (auto& x : th) x.join();
        uint64_t nb = 0, inst = 0, kr = 0; uint32_t mx = 0;
        for (unsigned t = 0; t < nt; ++t) {
            kr += t_kr[t];
            if (t_kind[t] == 1) W2R_FAIL(W2RAP_ERR_BAD_ARG, "read %llu: base offsets do not hold its bases", (unsigned long long)t_bad[t]);
            if (t_kind[t] == 2) W2R_FAIL(W2RAP_ERR_BAD_ARG, "read %llu: empty quality stream (at least the terminator byte is required)", (unsigned long long)t_bad[t]);
            nb += t_nb[t]; inst += t_inst[t]; mx = std::max(mx, t_mx[t]);
        }
        if (mx > 65535u) W2R_FAIL(W2RAP_ERR_BAD_ARG, "reads longer than 65535 bases are not supported (the reference stores good lengths in uint16_t)");
        d->n_bases = nb; d->max_len = mx; d->n_inst_upper = inst; d->n_kreads = kr;
    }
    const double t1 = now_ms();
    // +32 bytes of padding: packed bases are read with aligned 8-byte loads that may touch a few bytes past a read
    if (d->pooled) {        // host-buffer entry point: try to take the per-device arena
        UploadArena& a = UploadArena::get(device);
        std::lock_guard<std::mutex> g(a.mu);
        if (!a.in_use) { a.in_use = true; d->arena = true; }
    }
    dev_alloc(d, (void**)&d->bases, d->bases_bytes + 32, s, 0);
    dev_alloc(d, (void**)&d->quals, d->quals_bytes + 32, s, 1);
    dev_alloc(d, (void**)&d->base_off, (n + 1) * 8, s, 2);
    dev_alloc(d, (void**)&d->qual_off, (n + 1) * 8, s, 3);
    dev_alloc(d, (void**)&d->len, (n + 1) * 4, s, 4);
    W2R_CUDA(cudaMemsetAsync(d->bases + d->bases_bytes, 0, 32, s));
    W2R_CUDA(cudaMemsetAsync(d->quals + d->quals_bytes, 0, 32, s));
    const double t2 = now_ms();
    if (n) {
        const unsigned nbatch = forced_batches ? (unsigned)forced_batches : (batched && n >= (1u << 20)) ? 8u : 1u;
        for (unsigned b = 0; b < nbatch; ++b) {
            const uint64_t r0 = n * b / nbatch, r1 = n * (b + 1) / nbatch;
            const uint64_t b0 = in->base_off[r0], b1 = in->base_off[r1], q0 = in->qual_off[r0], q1 = in->qual_off[r1];
            W2R_CUDA(cudaMemcpyAsync(d->len + r0, in->len + r0, (r1 - r0) * 4, cudaMemcpyHostToDevice, s));
            W2R_CUDA(cudaMemcpyAsync(d->base_off + r0, in->base_off + r0, (r1 - r0 + 1) * 8, cudaMemcpyHostToDevice, s));
            W2R_CUDA(cudaMemcpyAsync(d->qual_off + r0, in->qual_off + r0, (r1 - r0 + 1) * 8, cudaMemcpyHostToDevice, s));
            W2R_CUDA(cudaMemcpyAsync(d->bases + b0, in->bases + b0, b1 - b0, cudaMemcpyHostToDevice, s));
            W2R_CUDA(cudaMemcpyAsync(d->quals + q0, in->quals + q0, q1 - q0, cudaMemcpyHostToDevice, s));
            if (batched) {
                cudaEvent_t e;
                W2R_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                W2R_CUDA(cudaEventRecord(e, s));
                d->batch_ready.push_back(e);
                d->batch_first.push_back(r0);
            }
        }
        if (batched) d->batch_first.push_back(n);
    } else {
        uint64_t z = 0;
        W2R_CUDA(cudaMemcpyAsync(d->base_off, &z, 8, cudaMemcpyHostToDevice, s));
        W2R_CUDA(cudaMemcpyAsync(d->qual_off, &z, 8, cudaMemcpyHostToDevice, s));
    }
    if (!batched) W2R_CUDA(cudaStreamSynchronize(s));
    if (getenv("W2RAP_TRACE")) fprintf(stderr, "[w2rap] upload: validate %.1f ms, alloc %.1f ms, enqueue %.1f ms\n", t1 - t0, t2 - t1, now_ms() - t2);
}

static void check_params(const w2rap_params* p) {
    if (!p) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null params");
    if (p->abi_version != W2RAP_STEP2_ABI_VERSION) W2R_FAIL(W2RAP_ERR_BAD_ARG, "ABI version %u, library has %d", p->abi_version, W2RAP_STEP2_ABI_VERSION);
    if (p->K != W2RAP_K) W2R_FAIL(W2RAP_ERR_BAD_ARG, "K=%u: only K=60 is built (the reference hard-wires it, BuildReadQGraph.cc:51)", p->K);
    if (p->min_freq == 0 || p->min_freq > 255) W2R_FAIL(W2RAP_ERR_BAD_ARG, "min_freq must be in 1..255 (counts saturate at 255)");
    if (p->force_passes > 4096) W2R_FAIL(W2RAP_ERR_BAD_ARG, "force_passes must be <= 4096");
    if (p->places_K2 && (p->places_K2 < W2RAP_K || !p->want_paths || !p->apply_fixpaths))
        W2R_FAIL(W2RAP_ERR_BAD_ARG, "places_K2 needs want_paths and apply_fixpaths (step 3 reads the paths after FixPaths) and K2 >= 60");
}

}  // namespace w2r

struct w2rap_comm { int world, rank, device; w2r::ncclComm_t comm; };

namespace w2r {
// count_into: w2rap_step2_count (the count stage alone, into the handle); build_from: w2rap_step2_build (select, then the rest)
static void run_on_device(DeviceReads& dr, const w2rap_params* p, w2rap_graph* out, float h2d_ms, const w2rap_comm* cm = nullptr, double t_entry = 0,
                          w2rap_counts* count_into = nullptr, const w2rap_counts* build_from = nullptr) {
    GraphOwner* owner = new GraphOwner();
    memset(out, 0, sizeof(*out));
    out->_owner = owner;
    try {
        { Ctx probe; check_device(dr.device, probe); }
        SlabLease lease(dr.device);                  // declared before the pipeline: its buffers go back before the lease does
        Pipeline pl(dr, *p, out, owner);
        if (cm) { pl.world = cm->world; pl.rank = cm->rank; pl.comm = cm->comm; }
        check_device(dr.device, pl.c);
        pl.c.slab = lease.slab;
        const double t_run = now_ms();
        pl.from_counts = build_from;
        if (count_into) pl.run_count(count_into); else pl.run();
        out->timings.h2d_ms = h2d_ms;
        out->timings.total_ms += h2d_ms;
        out->timings.host_pre_ms = t_entry ? (float)(t_run - t_entry) : 0.f;
        out->timings.wall_ms = (float)(now_ms() - (t_entry ? t_entry : t_run));
    } catch (...) {
        delete owner;
        memset(out, 0, sizeof(*out));
        throw;
    }
}

// Which calls a counts handle may go to: a sharded count only to the sharded calls with its own communicator (every rank holds
// only its partitions), a single-GPU count only to the single-GPU calls.  Shared by every entry point that takes a handle.
static void check_counts_comm(const w2rap_counts* h, const w2rap_comm* comm) {
    if (h->comm && !comm) W2R_FAIL(W2RAP_ERR_BAD_ARG, "these counts are sharded (w2rap_step2_count_sharded): they hold this rank's partitions only; use the _sharded calls");
    if (!h->comm && comm) W2R_FAIL(W2RAP_ERR_BAD_ARG, "these counts were made on one GPU (w2rap_step2_count): use the single-GPU calls");
    if (h->comm != comm) W2R_FAIL(W2RAP_ERR_BAD_ARG, "these counts were made with another communicator: use the one they were counted with");
}

// The argument checks of a count, on one GPU (sharded = false, comm unused) or sharded.  Made before any device work or collective.
static void check_count_args(const w2rap_device_reads* reads, const w2rap_params* p, w2rap_counts** counts, const w2rap_comm* comm, bool sharded) {
    if (!reads || !counts || (sharded && !comm)) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null argument");
    *counts = nullptr;
    check_params(p);
    if (sharded && p->dump_kmers) W2R_FAIL(W2RAP_ERR_BAD_ARG, "dump_kmers must be 0 for a sharded count (level 2 is a single-GPU test hook, level 1 dumps the dictionary of a build)");
    if (p->dump_kmers == 1) W2R_FAIL(W2RAP_ERR_BAD_ARG, "dump_kmers 1 dumps the solid dictionary, which only a build makes: a count takes dump_kmers 0 or 2");
    if (p->dump_kmers > 2) W2R_FAIL(W2RAP_ERR_BAD_ARG, "dump_kmers must be 0 or 2 for a count");
    if (sharded && reads->d.device != comm->device) W2R_FAIL(W2RAP_ERR_BAD_ARG, "read shard lives on device %d, communicator on %d", reads->d.device, comm->device);
}

// The argument checks of a build, on one GPU (comm = null) or sharded.  Made before any device work or collective.
static void check_build_args(const w2rap_device_reads* reads, const w2rap_counts* counts, const w2rap_params* p, const w2rap_graph* out, const w2rap_comm* comm,
                             bool sharded) {
    if (!reads || !counts || !out || (sharded && !comm)) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null argument");
    check_params(p);
    check_counts_comm(counts, comm);
    if (p->min_freq < counts->f0)
        W2R_FAIL(W2RAP_ERR_BAD_ARG, "min_freq %u is below the keep floor %u of these counts (k-mers seen fewer times were not kept): count again with min_freq <= %u",
                 p->min_freq, counts->f0, p->min_freq);
    if (p->min_qual != counts->min_qual)
        W2R_FAIL(W2RAP_ERR_BAD_ARG, "min_qual %u differs from the min_qual %u these counts were made with (the quality floor changes the counts): count again",
                 p->min_qual, counts->min_qual);
    if (p->dump_kmers == 2) W2R_FAIL(W2RAP_ERR_BAD_ARG, "dump_kmers 2 (every distinct k-mer with its count) comes from w2rap_step2_count, not from a build");
    if (p->dump_kmers > 2) W2R_FAIL(W2RAP_ERR_BAD_ARG, "dump_kmers must be 0 or 1 for a build");
    if (reads != counts->reads || reads->d.n != counts->n_reads || reads->d.n_bases != counts->n_bases)
        W2R_FAIL(W2RAP_ERR_BAD_ARG, "the reads handle is not the one these counts were made from: a build paths the reads that were counted");
}

// w2rap_step2_count(_sharded) after the checks: the count stage into a new handle, and <workdir>/small_K.freqs from rank 0.
static int count_into_handle(w2rap_device_reads* reads, const w2rap_params* p, const w2rap_comm* comm, w2rap_counts** counts, w2rap_graph* summary,
                             char* err, size_t errlen) {
    w2rap_counts* h = new w2rap_counts();
    h->reads = reads; h->n_reads = reads->d.n; h->n_bases = reads->d.n_bases; h->device = reads->d.device;
    h->min_qual = p->min_qual; h->f0 = p->min_freq;
    if (comm) { h->comm = comm; h->world = comm->world; h->rank = comm->rank; }
    w2rap_graph local;
    w2rap_graph* out = summary ? summary : &local;
    try {
        run_on_device(reads->d, p, out, 0.f, comm, 0, h);
    } catch (...) { w2rap_step2_counts_release(h); throw; }
    int rc = W2RAP_OK;
    if (h->rank == 0 && p->workdir && p->workdir[0]) { std::string f = std::string(p->workdir) + "/small_K.freqs"; rc = w2rap_write_freqs(f.c_str(), out, err, errlen); }
    if (!summary) w2rap_step2_free(&local);
    if (rc) { w2rap_step2_counts_release(h); return rc; }
    *counts = h;
    return W2RAP_OK;
}

}  // namespace w2r

// ================================================================ C ABI
using namespace w2r;

static int fail(const Error& e, char* err, size_t errlen) {
    if (err && errlen) { snprintf(err, errlen, "%s", e.msg.c_str()); }
    return e.code;
}
#define W2R_API_BEGIN try {
#define W2R_API_END                                                                                                  \
    }                                                                                                                \
    catch (const Error& e) { return fail(e, err, errlen); }                                                          \
    catch (const std::exception& e) { return fail(Error{W2RAP_ERR_INTERNAL, e.what()}, err, errlen); }               \
    return W2RAP_OK;

extern "C" {

int w2rap_step2_abi_version(void) { return W2RAP_STEP2_ABI_VERSION; }
const char* w2rap_step2_build_info(void) { return "w2rap step2 B200 (sm_100a), K=60, built " __DATE__ " " __TIME__; }

int w2rap_step2_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n; ++i) { cudaDeviceProp pr; if (cudaGetDeviceProperties(&pr, i) == cudaSuccess && pr.major >= 10) ++ok; }
    return ok;
}

int w2rap_step2_upload(const w2rap_reads* in, int device, w2rap_device_reads** handle, char* err, size_t errlen) {
    W2R_API_BEGIN
    if (!handle) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null handle");
    validate_reads(in);
    Ctx c; check_device(device, c);
    w2rap_device_reads* h = new w2rap_device_reads();
    try { upload(in, c.device, &h->d, 0, false); } catch (...) { h->d.release(); delete h; throw; }
    *handle = h;
    W2R_API_END
}

void w2rap_step2_release(w2rap_device_reads* handle) {
    if (!handle) return;
    cudaSetDevice(handle->d.device);
    handle->d.release();
    delete handle;
}

int w2rap_step2_run_resident(w2rap_device_reads* handle, const w2rap_params* p, w2rap_graph* out, char* err, size_t errlen) {
    W2R_API_BEGIN
    if (!handle || !out) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null argument");
    check_params(p);
    run_on_device(handle->d, p, out, 0.f);
    if (p->workdir && p->workdir[0]) { std::string f = std::string(p->workdir) + "/small_K.freqs"; int rc = w2rap_write_freqs(f.c_str(), out, err, errlen); if (rc) return rc; }
    W2R_API_END
}

int w2rap_step2_run(const w2rap_reads* in, const w2rap_params* p, w2rap_graph* out, char* err, size_t errlen) {
    W2R_API_BEGIN
    const double t_entry = now_ms();
    if (!out) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null output");
    check_params(p);
    validate_reads(in);
    Ctx c; check_device(p->device, c);
    DeviceReads d;
    d.pooled = true;
    cudaStream_t us = nullptr;
    W2R_CUDA(cudaStreamCreateWithFlags(&us, cudaStreamNonBlocking));
    d.pool_stream = us;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    float h2d = 0;
    try {
        cudaEventRecord(e0, us);
        upload(in, c.device, &d, us, true);
        cudaEventRecord(e1, us);
        run_on_device(d, p, out, 0.f, nullptr, t_entry);          // consumes the batches as they land
        cudaEventSynchronize(e1); cudaEventElapsedTime(&h2d, e0, e1);
        out->timings.h2d_ms = h2d;              // overlapped with the quality floor + extraction, already inside total_ms
    } catch (...) { cudaStreamSynchronize(us); d.release(); cudaStreamDestroy(us); cudaEventDestroy(e0); cudaEventDestroy(e1); throw; }
    const double t_post = now_ms();
    cudaStreamSynchronize(us); d.release(); cudaStreamDestroy(us); cudaEventDestroy(e0); cudaEventDestroy(e1);
    out->timings.host_post_ms = (float)(now_ms() - t_post);
    out->timings.wall_ms = (float)(now_ms() - t_entry);
    if (p->workdir && p->workdir[0]) { std::string f = std::string(p->workdir) + "/small_K.freqs"; int rc = w2rap_write_freqs(f.c_str(), out, err, errlen); if (rc) return rc; }
    W2R_API_END
}

int w2rap_step2_comm_unique_id(uint8_t* id128, char* err, size_t errlen) {
    W2R_API_BEGIN
    if (!id128) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null id buffer");
    NcclApi& n = NcclApi::get();
    if (n.error) W2R_FAIL(W2RAP_ERR_NO_DEVICE, "%s", n.error);
    ncclUniqueId id;
    if (n.GetUniqueId(&id) != ncclSuccess) W2R_FAIL(W2RAP_ERR_CUDA, "ncclGetUniqueId failed");
    memcpy(id128, id.internal, 128);
    W2R_API_END
}

int w2rap_step2_comm_init(const uint8_t* id128, int world, int rank, int device, w2rap_comm** comm, char* err, size_t errlen) {
    W2R_API_BEGIN
    if (!id128 || !comm || world < 1 || rank < 0 || rank >= world) W2R_FAIL(W2RAP_ERR_BAD_ARG, "bad communicator arguments");
    if (world & (world - 1)) W2R_FAIL(W2RAP_ERR_BAD_ARG, "world size must be a power of two (partition ranges are split evenly)");
    NcclApi& n = NcclApi::get();
    if (n.error) W2R_FAIL(W2RAP_ERR_NO_DEVICE, "%s", n.error);
    Ctx c; check_device(device, c);
    ncclUniqueId id;
    memcpy(id.internal, id128, 128);
    ncclComm_t nc = nullptr;
    ncclResult_t r = n.CommInitRank(&nc, world, id, rank);
    if (r != ncclSuccess) W2R_FAIL(W2RAP_ERR_CUDA, "ncclCommInitRank failed: %s", n.GetErrorString(r));
    *comm = new w2rap_comm{world, rank, c.device, nc};
    W2R_API_END
}

void w2rap_step2_comm_destroy(w2rap_comm* comm) {
    if (!comm) return;
    cudaSetDevice(comm->device);
    if (comm->comm) NcclApi::get().CommDestroy(comm->comm);
    delete comm;
}

int w2rap_step2_run_sharded_resident(w2rap_device_reads* handle, const w2rap_params* p, w2rap_comm* comm, w2rap_graph* out, char* err, size_t errlen) {
    W2R_API_BEGIN
    if (!handle || !out || !comm) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null argument");
    check_params(p);
    if (handle->d.device != comm->device) W2R_FAIL(W2RAP_ERR_BAD_ARG, "read shard lives on device %d, communicator on %d", handle->d.device, comm->device);
    run_on_device(handle->d, p, out, 0.f, comm);
    if (comm->rank == 0 && p->workdir && p->workdir[0]) { std::string f = std::string(p->workdir) + "/small_K.freqs"; int rc = w2rap_write_freqs(f.c_str(), out, err, errlen); if (rc) return rc; }
    W2R_API_END
}

int w2rap_step2_run_sharded(const w2rap_reads* shard, const w2rap_params* p, w2rap_comm* comm, w2rap_graph* out, char* err, size_t errlen) {
    W2R_API_BEGIN
    if (!out || !comm) W2R_FAIL(W2RAP_ERR_BAD_ARG, "null argument");
    check_params(p);
    validate_reads(shard);
    Ctx c; check_device(comm->device, c);
    DeviceReads d;
    d.pooled = true;
    cudaStream_t us = nullptr;
    W2R_CUDA(cudaStreamCreateWithFlags(&us, cudaStreamNonBlocking));
    d.pool_stream = us;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    float h2d = 0;
    try {
        cudaEventRecord(e0, us);
        upload(shard, c.device, &d, us, true);
        cudaEventRecord(e1, us);
        run_on_device(d, p, out, 0.f, comm);
        cudaEventSynchronize(e1); cudaEventElapsedTime(&h2d, e0, e1);
        out->timings.h2d_ms = h2d;
    } catch (...) { cudaStreamSynchronize(us); d.release(); cudaStreamDestroy(us); cudaEventDestroy(e0); cudaEventDestroy(e1); throw; }
    cudaStreamSynchronize(us); d.release(); cudaStreamDestroy(us); cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (comm->rank == 0 && p->workdir && p->workdir[0]) { std::string f = std::string(p->workdir) + "/small_K.freqs"; int rc = w2rap_write_freqs(f.c_str(), out, err, errlen); if (rc) return rc; }
    W2R_API_END
}

// ---- count once, build for several min_freq (include/w2rap_step2_counts.h, include/w2rap_step2_counts_sharded.h)
int w2rap_step2_count(w2rap_device_reads* reads, const w2rap_params* p, w2rap_counts** counts, w2rap_graph* summary, char* err, size_t errlen) {
    W2R_API_BEGIN
    check_count_args(reads, p, counts, nullptr, false);
    if (int rc = count_into_handle(reads, p, nullptr, counts, summary, err, errlen)) return rc;
    W2R_API_END
}

int w2rap_step2_count_sharded(w2rap_device_reads* shard, const w2rap_params* p, w2rap_comm* comm, w2rap_counts** counts, w2rap_graph* summary, char* err, size_t errlen) {
    W2R_API_BEGIN
    check_count_args(shard, p, counts, comm, true);
    if (int rc = count_into_handle(shard, p, comm, counts, summary, err, errlen)) return rc;
    W2R_API_END
}

int w2rap_step2_build(w2rap_device_reads* reads, const w2rap_counts* counts, const w2rap_params* p, w2rap_graph* out, char* err, size_t errlen) {
    W2R_API_BEGIN
    check_build_args(reads, counts, p, out, nullptr, false);
    run_on_device(reads->d, p, out, 0.f, nullptr, 0, nullptr, counts);
    if (p->workdir && p->workdir[0]) { std::string f = std::string(p->workdir) + "/small_K.freqs"; int rc = w2rap_write_freqs(f.c_str(), out, err, errlen); if (rc) return rc; }
    W2R_API_END
}

int w2rap_step2_build_sharded(w2rap_device_reads* shard, const w2rap_counts* counts, const w2rap_params* p, w2rap_comm* comm, w2rap_graph* out, char* err, size_t errlen) {
    W2R_API_BEGIN
    check_build_args(shard, counts, p, out, comm, true);
    run_on_device(shard->d, p, out, 0.f, comm, 0, nullptr, counts);
    if (comm->rank == 0 && p->workdir && p->workdir[0]) { std::string f = std::string(p->workdir) + "/small_K.freqs"; int rc = w2rap_write_freqs(f.c_str(), out, err, errlen); if (rc) return rc; }
    W2R_API_END
}

void w2rap_step2_counts_release(w2rap_counts* counts) {
    if (!counts) return;
    cudaSetDevice(counts->device);
    // (stream-ordered allocations: every call that used them has drained its stream before returning)
    if (counts->solid) cudaFreeAsync(counts->solid, 0);
    if (counts->count) cudaFreeAsync(counts->count, 0);
    cudaStreamSynchronize(0);
    cudaGetLastError();
    delete counts;
}

void* w2rap_step2_host_alloc(size_t bytes) {
    try { return PinnedPool::get().acquire(bytes); } catch (...) { cudaGetLastError(); return nullptr; }
}
void w2rap_step2_host_free(void* p) { if (p) PinnedPool::get().release(p); }

void w2rap_step2_free(w2rap_graph* out) {
    if (!out) return;
    delete (GraphOwner*)out->_owner;
    memset(out, 0, sizeof(*out));
}

}  // extern "C"
