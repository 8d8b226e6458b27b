// Multi-GPU batch and NUMA-aware page-locked host buffers (include/pvgpu.h: pvgpu_mbatch_*, pvgpu_host_*).
//
// The reference is single-threaded and single-device; "4096 streams sharded across 1/2/4/8 B200" (BASELINE.json
// configs[3]) is new work (SURVEY 8(e)): streams are independent, so the batch is partitioned by stream, every device
// runs its own pvgpu_batch from its own host thread, and the only "gather" is each device's D2H copy landing in the
// caller's row pointers.  No collective, no peer traffic.
//
// Host side of the copies: a B200 box has two CPU sockets; pinned memory that lives on the other socket than the GPU
// crosses the inter-socket link and halves the copy rate when all eight GPUs move data at once.  pvgpu_host_alloc places
// the pages on the GPU's own NUMA node (mbind) -- optionally on explicit 2 MB huge pages -- before registering them with
// CUDA, and the worker thread of a device runs on that node's cores.
#include <cuda_runtime_api.h>
#include <sched.h>
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <cerrno>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pvgpu.h"
#include "pv_internal.h"
#include "pv_plan.h"

#if defined(__x86_64__)
#include <emmintrin.h>
#endif

namespace pvgpu {

// ---- NUMA placement without libnuma -------------------------------------------------------------------------------
// node of a CUDA device from sysfs (/sys/bus/pci/devices/<domain:bus:dev.fn>/numa_node); -1 when unknown
static int device_numa_node(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char *c = bus; *c; ++c) *c = (char)tolower(*c);
    const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
    FILE *f = fopen(path.c_str(), "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

// cpus of a node from /sys/devices/system/node/node<N>/cpulist ("0-47,96-143")
static bool node_cpuset(int node, cpu_set_t *set) {
    char path[96];
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    FILE *f = fopen(path, "r");
    if (!f) return false;
    char buf[4096] = {0};
    const bool ok = fgets(buf, sizeof buf, f) != nullptr;
    fclose(f);
    if (!ok) return false;
    CPU_ZERO(set);
    int n = 0;
    for (char *tok = strtok(buf, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a = 0, b = 0;
        if (sscanf(tok, "%d-%d", &a, &b) == 2) { for (int c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET(c, set); ++n; } }
        else if (sscanf(tok, "%d", &a) == 1 && a < CPU_SETSIZE) { CPU_SET(a, set); ++n; }
    }
    return n > 0;
}

// run the calling thread on the cores of `device`'s node (no-op when the topology is not visible)
static void bind_thread_to_device_node(int device) {
    const int node = device_numa_node(device);
    cpu_set_t set;
    if (node >= 0 && node_cpuset(node, &set)) sched_setaffinity(0, sizeof set, &set);
}

static long mbind_node(void *p, size_t bytes, int node) {
#ifdef SYS_mbind
    if (node < 0 || node >= 64) return -1;
    unsigned long mask = 1ul << node;
    const int kBind = 2 /* MPOL_BIND */;
    return syscall(SYS_mbind, p, bytes, kBind, &mask, (unsigned long)(8 * sizeof mask), 0u);
#else
    (void)p; (void)bytes; (void)node;
    return -1;
#endif
}

struct HostBlock { size_t bytes; bool mapped; int node; bool huge; };
static std::mutex g_host_mu;
static std::map<void *, HostBlock> g_host_blocks;

}  // namespace pvgpu

using namespace pvgpu;

// ------------------------------------------------------------------------------------------------
// multi-device batch
// ------------------------------------------------------------------------------------------------
struct pvgpu_mbatch {
    pvgpu_config cfg{};
    int n_streams = 0, channels = 1;
    std::vector<int> devices;
    std::vector<pvgpu_batch *> parts;           // one per device (null when the device got no stream)
    std::vector<std::vector<int>> members;      // stream indices of every device, ascending
    std::vector<int> owner;
    std::vector<int64_t> n_in, n_out;
    bool planned = false;
    ~pvgpu_mbatch() { for (auto *b : parts) if (b) pvgpu_batch_destroy(b); }
};

// run fn(d) for every device index on its own thread; returns the first failure (message moved to the caller's thread)
template <class Fn> static int for_each_device(pvgpu_mbatch *m, Fn fn) {
    const int nd = (int)m->devices.size();
    std::vector<int> rc(nd, PVGPU_OK);
    std::vector<std::string> msg(nd);
    std::vector<std::thread> th;
    th.reserve(nd);
    for (int d = 0; d < nd; ++d)
        th.emplace_back([&, d]() {
            bind_thread_to_device_node(m->devices[d]);
            try {   // an exception must neither leave the thread nor cross the C ABI
                rc[d] = fn(d);
                if (rc[d] != PVGPU_OK) msg[d] = last_error_string();
            } catch (const std::bad_alloc &) {
                rc[d] = PVGPU_ENOMEM; msg[d] = "out of host memory";
            } catch (...) {
                rc[d] = PVGPU_ESTATE; msg[d] = "unexpected failure";
            }
        });
    for (auto &t : th) t.join();
    for (int d = 0; d < nd; ++d)
        if (rc[d] != PVGPU_OK) return fail(rc[d], "device %d: %s", m->devices[d], msg[d].c_str());
    return PVGPU_OK;
}

extern "C" {

int pvgpu_shard_streams(const int64_t *n_in, int n_streams, int n_dev, int *owner) {
    if (!n_in || !owner || n_streams < 0 || n_dev < 1) return fail(PVGPU_EINVAL, "bad argument");
    partition_streams(n_in, n_streams, n_dev, owner);
    return PVGPU_OK;
}

int pvgpu_mbatch_create(const pvgpu_config *cfg, int n_streams, int64_t max_in_samples, const int *devices, int n_dev, pvgpu_mbatch **out) {
    if (!cfg || !out || n_streams < 1 || max_in_samples < 0) return fail(PVGPU_EINVAL, "bad batch arguments");
    const int visible = pvgpu_device_count();
    if (visible < 1) return fail(PVGPU_ECUDA, "no CUDA device: the phase vocoder has no CPU fallback");
    std::unique_ptr<pvgpu_mbatch> m(new (std::nothrow) pvgpu_mbatch);
    if (!m) return fail(PVGPU_ENOMEM, "out of host memory");
    m->cfg = *cfg;
    m->n_streams = n_streams;
    m->channels = cfg->channels;
    if (devices && n_dev > 0) m->devices.assign(devices, devices + n_dev);
    else for (int d = 0; d < visible; ++d) m->devices.push_back(d);      // devices == NULL: every visible device
    for (size_t i = 0; i < m->devices.size(); ++i) {
        if (m->devices[i] < 0 || m->devices[i] >= visible) return fail(PVGPU_EINVAL, "device %d out of range (%d devices)", m->devices[i], visible);
        for (size_t j = 0; j < i; ++j) if (m->devices[j] == m->devices[i]) return fail(PVGPU_EINVAL, "device %d listed twice", m->devices[i]);
    }
    m->parts.assign(m->devices.size(), nullptr);
    m->members.resize(m->devices.size());
    // the per-device batches are created by pvgpu_mbatch_plan, once the lengths (and so the partition) are known; the
    // configuration is validated now
    pvgpu_info info;
    int rc = pvgpu_describe(cfg, &info);
    if (rc) return rc;
    m->n_in.assign(n_streams, max_in_samples);
    *out = m.release();
    return PVGPU_OK;
}

void pvgpu_mbatch_destroy(pvgpu_mbatch *m) { delete m; }

int pvgpu_mbatch_plan(pvgpu_mbatch *m, const int64_t *n_in, int block, int64_t *n_out) {
    if (!m || !n_in) return fail(PVGPU_EINVAL, "null argument");
    const int nd = (int)m->devices.size();
    int64_t max_in = 0;
    for (int s = 0; s < m->n_streams; ++s) { if (n_in[s] < 0) return fail(PVGPU_EINVAL, "stream %d: negative length", s); if (n_in[s] > max_in) max_in = n_in[s]; }
    m->owner.assign(m->n_streams, 0);
    partition_streams(n_in, m->n_streams, nd, m->owner.data());
    std::vector<std::vector<int>> members(nd);
    for (int s = 0; s < m->n_streams; ++s) members[m->owner[s]].push_back(s);
    m->n_in.assign(n_in, n_in + m->n_streams);
    m->n_out.assign(m->n_streams, 0);
    m->planned = false;
    const int rc = for_each_device(m, [&](int d) -> int {
        const std::vector<int> &mem = members[d];
        if (m->parts[d]) { pvgpu_batch_destroy(m->parts[d]); m->parts[d] = nullptr; }   // planning is not the hot path: start clean
        if (mem.empty()) return PVGPU_OK;
        int r;
        pvgpu_config c = m->cfg;
        c.device = m->devices[d];
        if ((r = pvgpu_batch_create(&c, (int)mem.size(), max_in, &m->parts[d]))) return r;
        std::vector<int64_t> li(mem.size()), lo(mem.size());
        for (size_t i = 0; i < mem.size(); ++i) li[i] = n_in[mem[i]];
        if ((r = pvgpu_batch_plan(m->parts[d], li.data(), block, lo.data()))) return r;
        for (size_t i = 0; i < mem.size(); ++i) m->n_out[mem[i]] = lo[i];
        return PVGPU_OK;
    });
    if (rc) return rc;
    m->members.swap(members);
    if (n_out) for (int s = 0; s < m->n_streams; ++s) n_out[s] = m->n_out[s];
    m->planned = true;
    return PVGPU_OK;
}

int pvgpu_mbatch_run_host(pvgpu_mbatch *m, const void *const *in_rows, void *const *out_rows, int fmt) {
    if (!m || !in_rows || !out_rows) return fail(PVGPU_EINVAL, "null argument");
    if (!m->planned) return fail(PVGPU_ESTATE, "pvgpu_mbatch_plan has not been called");
    const int C = m->channels;
    return for_each_device(m, [&](int d) -> int {
        const std::vector<int> &mem = m->members[d];
        if (mem.empty()) return PVGPU_OK;
        // the device's rows, in its own stream order; contiguous members keep evenly spaced rows evenly spaced, so the
        // time-sliced host pipeline of the single-device batch still applies
        std::vector<const void *> ir(mem.size() * C);
        std::vector<void *> orw(mem.size() * C);
        for (size_t i = 0; i < mem.size(); ++i)
            for (int c = 0; c < C; ++c) { ir[i * C + c] = in_rows[(size_t)mem[i] * C + c]; orw[i * C + c] = out_rows[(size_t)mem[i] * C + c]; }
        return pvgpu_batch_run_host(m->parts[d], ir.data(), orw.data(), fmt);
    });
}

int pvgpu_mbatch_stats(const pvgpu_mbatch *m, int64_t *kernel_launches, int64_t *h2d_bytes, int64_t *d2h_bytes, int *devices_used) {
    if (!m) return fail(PVGPU_EINVAL, "null batch");
    int64_t kl = 0, hi = 0, ho = 0;
    int used = 0;
    for (pvgpu_batch *b : m->parts) {
        if (!b) continue;
        int64_t a = 0, s = 0, x = 0, y = 0;
        pvgpu_batch_stats(b, &a, &s, &x, &y);
        kl += a; hi += x; ho += y; ++used;
    }
    if (kernel_launches) *kernel_launches = kl;
    if (h2d_bytes) *h2d_bytes = hi;
    if (d2h_bytes) *d2h_bytes = ho;
    if (devices_used) *devices_used = used;
    return PVGPU_OK;
}

int pvgpu_mbatch_owner(const pvgpu_mbatch *m, int *owner_device /*[n_streams]*/) {
    if (!m || !owner_device) return fail(PVGPU_EINVAL, "null argument");
    if (!m->planned) return fail(PVGPU_ESTATE, "pvgpu_mbatch_plan has not been called");
    for (int s = 0; s < m->n_streams; ++s) owner_device[s] = m->devices[m->owner[s]];
    return PVGPU_OK;
}

// ------------------------------------------------------------------------------------------------
// page-locked host buffers on the device's NUMA node
// ------------------------------------------------------------------------------------------------
int pvgpu_host_alloc(void **ptr, size_t bytes, int device, int flags) {
    if (!ptr || bytes == 0) return fail(PVGPU_EINVAL, "bad argument");
    *ptr = nullptr;
    if (pvgpu_device_count() < 1) return fail(PVGPU_ECUDA, "no CUDA device");
    const size_t two_mb = (size_t)2 << 20;
    const size_t len = (bytes + two_mb - 1) / two_mb * two_mb;
    const int node = device >= 0 ? device_numa_node(device) : -1;
    void *p = MAP_FAILED;
    bool huge = false;
    if (flags & PVGPU_HOST_HUGEPAGES) {
        p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS | MAP_HUGETLB, -1, 0);
        huge = p != MAP_FAILED;
    }
    if (p == MAP_FAILED) p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p == MAP_FAILED) return fail(PVGPU_ENOMEM, "mmap of %zu bytes failed: %s", len, strerror(errno));
    if (!huge) madvise(p, len, MADV_HUGEPAGE);   // transparent huge pages where the kernel grants them
    const bool bound = (flags & PVGPU_HOST_NUMA_LOCAL) && node >= 0 && mbind_node(p, len, node) == 0;
    {   // first touch from a thread on the right node (covers kernels that refuse mbind inside a container)
        std::thread t([&]() {
            if ((flags & PVGPU_HOST_NUMA_LOCAL) && device >= 0) bind_thread_to_device_node(device);
            volatile char *c = (volatile char *)p;
            for (size_t o = 0; o < len; o += 4096) c[o] = 0;
        });
        t.join();
    }
    const cudaError_t e = cudaHostRegister(p, len, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        munmap(p, len);
        return fail(PVGPU_ENOMEM, "cudaHostRegister of %zu bytes failed: %s", len, cudaGetErrorString(e));
    }
    {
        std::lock_guard<std::mutex> g(g_host_mu);
        g_host_blocks[p] = HostBlock{len, true, bound ? node : -1, huge};
    }
    *ptr = p;
    return PVGPU_OK;
}

int pvgpu_host_free(void *ptr) {
    if (!ptr) return PVGPU_OK;
    HostBlock blk{};
    {
        std::lock_guard<std::mutex> g(g_host_mu);
        auto it = g_host_blocks.find(ptr);
        if (it == g_host_blocks.end()) return fail(PVGPU_EINVAL, "pointer was not returned by pvgpu_host_alloc");
        blk = it->second;
        g_host_blocks.erase(it);
    }
    cudaHostUnregister(ptr);
    cudaGetLastError();
    munmap(ptr, blk.bytes);
    return PVGPU_OK;
}

int pvgpu_host_info(const void *ptr, int *numa_node, int *hugepages, size_t *bytes) {
    std::lock_guard<std::mutex> g(g_host_mu);
    auto it = g_host_blocks.find(const_cast<void *>(ptr));
    if (it == g_host_blocks.end()) return fail(PVGPU_EINVAL, "pointer was not returned by pvgpu_host_alloc");
    if (numa_node) *numa_node = it->second.node;
    if (hugepages) *hugepages = it->second.huge ? 1 : 0;
    if (bytes) *bytes = it->second.bytes;
    return PVGPU_OK;
}

int pvgpu_device_numa_node(int device) { return device_numa_node(device); }

int pvgpu_bind_thread_to_device(int device) {
    bind_thread_to_device_node(device);
    return PVGPU_OK;
}

}  // extern "C"

namespace pvgpu {
void copy_nt(float *dst, const float *src, size_t n) {
#if defined(__x86_64__)
    auto one = [&](size_t i) { int v; std::memcpy(&v, src + i, sizeof v); _mm_stream_si32(reinterpret_cast<int *>(dst + i), v); };
    size_t i = 0;
    while (i < n && ((uintptr_t)(dst + i) & 15)) one(i++);
    for (; i + 4 <= n; i += 4) _mm_stream_ps(dst + i, _mm_loadu_ps(src + i));
    for (; i < n; ++i) one(i);
#else
    std::memcpy(dst, src, sizeof(float) * n);
#endif
}
void copy_nt(int16_t *dst, const int16_t *src, size_t n) {
#if defined(__x86_64__)
    auto pair = [&](size_t i) { int v; std::memcpy(&v, src + i, sizeof v); _mm_stream_si32(reinterpret_cast<int *>(dst + i), v); };
    size_t i = 0;
    if (n && ((uintptr_t)dst & 2)) { dst[0] = src[0]; i = 1; }   // _mm_stream_si32 needs 4-byte alignment: one plain store first
    for (; i + 2 <= n && ((uintptr_t)(dst + i) & 15); i += 2) pair(i);
    for (; i + 8 <= n; i += 8) _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i), _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i)));
    for (; i + 2 <= n; i += 2) pair(i);
    if (i < n) dst[i] = src[i];   // an odd last sample
#else
    std::memcpy(dst, src, sizeof(int16_t) * n);
#endif
}
void copy_nt_fence() {
#if defined(__x86_64__)
    _mm_sfence();
#endif
}
}  // namespace pvgpu
