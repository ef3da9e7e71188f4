// cgl_api.cu -- error state, device queries, host-buffer entry points, IPC + halo helpers.
#include <cuda.h>
#include <stdarg.h>
#include <string.h>

#include <map>
#include <mutex>

#include "cgl_internal.cuh"

namespace cgl {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int sm_count()
{
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// Wait until *flag - seq >= 0 (acquire, system scope).  Bounded: a peer that died or never launched its side of
// the exchange raises the halo alarm word after g_wait_ns instead of hanging this GPU until a device reset.
__device__ __forceinline__ bool spin_until(const uint32_t *flag, uint32_t seq)
{
    uint32_t v, spins = 0;
    unsigned long long t0 = 0;
    do {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int32_t)(v - seq) >= 0) return true;
        __nanosleep(64);
        if (spins == 0) t0 = globaltimer_ns();
    } while ((++spins & 127u) != 0 || !wait_expired(t0, ALARM_HALO));
    raise_alarm(ALARM_HALO);
    return false;
}

// Whole halo exchange of one rank in ONE launch: CTA 0 talks to the upper neighbour, CTA 1 to the
// lower one.  Each pushes its strip into the neighbour's landing slot and publishes `seq`, then waits
// for the neighbour's strip of the same block and moves it into its own ghost rows.  Every rank
// pushes before it waits, so the ring cannot deadlock.
struct HaloSide {
    const uint4 *src;        // my boundary rows
    uint4 *peer_landing;     // neighbour's landing slot for them
    uint32_t *peer_flag;
    const uint32_t *my_flag; // set by that neighbour
    const uint4 *my_landing;
    uint4 *ghost;            // my ghost rows on that side
};

// HX_CTAS CTAs per direction, each moving one slice of the strip: push my slice into the neighbour's landing slot,
// count my arrival on the neighbour's counter (release), wait until the neighbour's HX_CTAS slices of the same
// block have arrived on mine (acquire), move my slice of its strip into my ghost rows.  (One CTA per direction
// took ~15 us for the 512 KiB strips of C4; the exchange sits on the compute stream between two blocks.)
constexpr int HX_CTAS = 8;

__global__ void __launch_bounds__(1024) halo_exchange_kernel(HaloSide up, HaloSide dn, uint64_t n_vec, uint32_t uses)
{
    const HaloSide s = blockIdx.x < HX_CTAS ? up : dn;
    const uint32_t part = blockIdx.x % HX_CTAS;
    const uint64_t per = (n_vec + HX_CTAS - 1) / HX_CTAS;
    const uint64_t lo = part * per, hi = lo + per < n_vec ? lo + per : n_vec;
    for (uint64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) s.peer_landing[i] = s.src[i];
    __threadfence_system();
    __syncthreads();
    __shared__ int arrived;
    if (threadIdx.x == 0) {
        __threadfence_system();
        asm volatile("red.release.sys.global.add.u32 [%0], 1;" ::"l"(s.peer_flag) : "memory");
        arrived = spin_until(s.my_flag, uses * HX_CTAS);
    }
    __syncthreads();
    if (!arrived) return;                       // timed out: alarm raised, nothing copied from the landing zone
    for (uint64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) s.ghost[i] = __ldcg(s.my_landing + i);
}

CGL_DEFINE_TU_HOOKS(api)

// ---- alarm words + wait bound (see cgl_internal.cuh) ------------------------------------------------------
static int *g_alarm_host = nullptr, *g_alarm_dev = nullptr;
static unsigned long long g_wait_ns_host = 2000000000ull;
static bool g_hooks_set[64] = {};

static int apply_hooks()
{
    int rc;
    if ((rc = set_hooks_env(g_alarm_dev, g_wait_ns_host))) return rc;
    if ((rc = set_hooks_life_tb(g_alarm_dev, g_wait_ns_host))) return rc;
    return set_hooks_api(g_alarm_dev, g_wait_ns_host);
}

}  // namespace cgl

using namespace cgl;

extern "C" int cgl_alarm_words(int **host_words_out)
{
    CGL_REQUIRE(host_words_out, CGL_E_BADARG, "cgl_alarm_words: null");
    if (g_alarm_host == nullptr) {
        void *h = nullptr, *d = nullptr;
        CGL_CUDA(cudaHostAlloc(&h, CGL_ALARM_WORDS * sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
        memset(h, 0, CGL_ALARM_WORDS * sizeof(int));
        CGL_CUDA(cudaHostGetDevicePointer(&d, h, 0));
        g_alarm_host = static_cast<int *>(h);
        g_alarm_dev = static_cast<int *>(d);
    }
    int dev = 0;
    CGL_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !g_hooks_set[dev]) {
        int rc = apply_hooks();
        if (rc) return rc;
        g_hooks_set[dev] = true;
    }
    *host_words_out = g_alarm_host;
    return 0;
}

extern "C" int cgl_set_wait_timeout_ms(uint32_t ms)
{
    g_wait_ns_host = (unsigned long long)ms * 1000000ull;
    int dev = 0;
    CGL_CUDA(cudaGetDevice(&dev));
    int rc = apply_hooks();                         // current device now; other devices at their next cgl_alarm_words
    for (int i = 0; i < 64; ++i) g_hooks_set[i] = false;
    if (rc == 0 && dev >= 0 && dev < 64) g_hooks_set[dev] = true;
    return rc;
}

extern "C" int cgl_halo_exchange(const uint32_t *top_src, const uint32_t *bot_src, uint32_t *peer_up_landing,
                                 uint32_t *peer_dn_landing, uint32_t *peer_up_flag, uint32_t *peer_dn_flag,
                                 const uint32_t *my_landing_up, const uint32_t *my_landing_dn,
                                 const uint32_t *my_flag_up, const uint32_t *my_flag_dn, uint32_t *ghost_up,
                                 uint32_t *ghost_dn, uint64_t n_words, uint32_t seq, cgl_stream_t stream)
{
    CGL_REQUIRE(top_src && bot_src && peer_up_landing && peer_dn_landing && peer_up_flag && peer_dn_flag &&
                my_landing_up && my_landing_dn && my_flag_up && my_flag_dn && ghost_up && ghost_dn && n_words &&
                n_words % 4 == 0, CGL_E_BADARG, "cgl_halo_exchange: bad argument");
    HaloSide up{reinterpret_cast<const uint4 *>(top_src), reinterpret_cast<uint4 *>(peer_up_landing), peer_up_flag,
                my_flag_up, reinterpret_cast<const uint4 *>(my_landing_up), reinterpret_cast<uint4 *>(ghost_up)};
    HaloSide dn{reinterpret_cast<const uint4 *>(bot_src), reinterpret_cast<uint4 *>(peer_dn_landing), peer_dn_flag,
                my_flag_dn, reinterpret_cast<const uint4 *>(my_landing_dn), reinterpret_cast<uint4 *>(ghost_dn)};
    // `seq` = 1, 2, 3, ... per exchange; the two landing slots (and their counters) alternate, so this is use number
    // (seq + 1) / 2 of its slot
    halo_exchange_kernel<<<2 * HX_CTAS, 1024, 0, as_stream(stream)>>>(up, dn, n_words / 4, (seq + 1u) >> 1);
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_abi_version(void) { return CGL_B200_ABI_VERSION; }
extern "C" const char *cgl_last_error(void) { return g_err; }

extern "C" int cgl_device_count(int *count_out)
{
    CGL_REQUIRE(count_out, CGL_E_BADARG, "cgl_device_count: null");
    CGL_CUDA(cudaGetDeviceCount(count_out));
    return 0;
}

extern "C" int cgl_device_info(int device, char *name_out, int name_cap, int *sm_count_out,
                               int *cc_major_out, int *cc_minor_out, uint64_t *total_mem_out)
{
    cudaDeviceProp p;
    CGL_CUDA(cudaGetDeviceProperties(&p, device));
    if (name_out && name_cap > 0) {
        strncpy(name_out, p.name, (size_t)name_cap - 1);
        name_out[name_cap - 1] = 0;
    }
    if (sm_count_out) *sm_count_out = p.multiProcessorCount;
    if (cc_major_out) *cc_major_out = p.major;
    if (cc_minor_out) *cc_minor_out = p.minor;
    if (total_mem_out) *total_mem_out = (uint64_t)p.totalGlobalMem;
    return 0;
}

// ---- sim.__step_state_gpu replacement (CGL/CGL.py:203-208) --------------------------------
namespace {
struct HostStepScratch {
    uint64_t size = 0;
    uint8_t *cells = nullptr;
    int8_t *stable = nullptr;
    uint32_t *wa = nullptr, *wb = nullptr;
    int device = -1;
};
thread_local HostStepScratch g_hs;

int ensure_scratch(uint64_t size, uint32_t side)
{
    int dev = 0;
    CGL_CUDA(cudaGetDevice(&dev));
    if (g_hs.size >= size && g_hs.device == dev) return 0;
    if (g_hs.cells) { cudaFree(g_hs.cells); cudaFree(g_hs.stable); cudaFree(g_hs.wa); cudaFree(g_hs.wb); }
    g_hs = HostStepScratch();
    const uint64_t words = (uint64_t)side * cgl_words_per_row(side);
    CGL_CUDA(cudaMalloc(&g_hs.cells, size));
    CGL_CUDA(cudaMalloc(&g_hs.stable, size));
    CGL_CUDA(cudaMalloc(&g_hs.wa, words * 4));
    CGL_CUDA(cudaMalloc(&g_hs.wb, words * 4));
    g_hs.size = size;
    g_hs.device = dev;
    return 0;
}
}  // namespace

extern "C" int cgl_step_state_gpu(uint8_t *world_host, int8_t *stable_host, uint32_t side, int spawn,
                                  int stable_max)
{
    CGL_REQUIRE(world_host && stable_host && side, CGL_E_BADARG, "cgl_step_state_gpu: bad argument");
    const uint64_t size = (uint64_t)side * side;
    int rc = ensure_scratch(size, side);
    if (rc) return rc;
    cudaStream_t st = 0;
    CGL_CUDA(cudaMemcpyAsync(g_hs.cells, world_host, size, cudaMemcpyHostToDevice, st));
    CGL_CUDA(cudaMemcpyAsync(g_hs.stable, stable_host, size, cudaMemcpyHostToDevice, st));
    if ((rc = cgl_pack(g_hs.cells, g_hs.wa, 1, side, side, st))) return rc;
    if ((rc = cgl_env_step(g_hs.wa, g_hs.wb, g_hs.stable, 1, side, nullptr, spawn, stable_max, nullptr,
                           nullptr, nullptr, st)))
        return rc;
    if ((rc = cgl_unpack(g_hs.wb, g_hs.cells, 1, side, side, st))) return rc;
    CGL_CUDA(cudaMemcpyAsync(world_host, g_hs.cells, size, cudaMemcpyDeviceToHost, st));
    CGL_CUDA(cudaMemcpyAsync(stable_host, g_hs.stable, size, cudaMemcpyDeviceToHost, st));
    CGL_CUDA(cudaStreamSynchronize(st));
    return 0;
}

static int env_step_host_impl(uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs,
                              uint32_t side, const int32_t *actions_host, int32_t *actions_dev,
                              int spawn, int stable_max, int32_t *reward_dev, int32_t *reward_host,
                              int8_t *obs_host, cgl_stream_t stream, bool sync)
{
    CGL_REQUIRE(win && wout && stable && n_envs && side, CGL_E_BADARG, "cgl_env_step_host: bad argument");
    CGL_REQUIRE(!actions_host || actions_dev, CGL_E_BADARG, "cgl_env_step_host: actions scratch missing");
    CGL_REQUIRE(!reward_host || reward_dev, CGL_E_BADARG, "cgl_env_step_host: reward scratch missing");
    cudaStream_t st = as_stream(stream);
    if (actions_host)
        CGL_CUDA(cudaMemcpyAsync(actions_dev, actions_host, n_envs * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    // Pinned (device-mapped) reward buffer: the kernel writes the per-env rewards straight into host
    // memory (posted PCIe writes, 4 B per env) instead of a separate device-to-host copy.
    int32_t *reward_target = reward_host ? reward_dev : nullptr;
    bool reward_direct = false;
    if (reward_host) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, reward_host) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
            attr.devicePointer != nullptr) {
            reward_target = static_cast<int32_t *>(attr.devicePointer);
            reward_direct = true;
        } else {
            cudaGetLastError();          // pageable memory: clear the sticky "invalid value" and copy instead
        }
    }
    int rc = cgl_env_step(win, wout, stable, n_envs, side, actions_host ? actions_dev : nullptr, spawn,
                          stable_max, reward_target, nullptr, nullptr, stream);
    if (rc) return rc;
    if (reward_host && !reward_direct)
        CGL_CUDA(cudaMemcpyAsync(reward_host, reward_dev, n_envs * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (obs_host)
        CGL_CUDA(cudaMemcpyAsync(obs_host, stable, n_envs * (uint64_t)side * side, cudaMemcpyDeviceToHost, st));
    if (sync) CGL_CUDA(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int cgl_env_step_host(uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs,
                                 uint32_t side, const int32_t *actions_host, int32_t *actions_dev,
                                 int spawn, int stable_max, int32_t *reward_dev, int32_t *reward_host,
                                 int8_t *obs_host, cgl_stream_t stream)
{
    return env_step_host_impl(win, wout, stable, n_envs, side, actions_host, actions_dev, spawn, stable_max,
                              reward_dev, reward_host, obs_host, stream, true);
}

// Same, without the final synchronisation: the caller waits with cgl_stream_wait (or any stream sync) before it
// reads reward_host / obs_host or overwrites actions_host.  Two env groups on two streams then overlap one
// group's host round trip with the other group's step.
extern "C" int cgl_env_step_host_async(uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs,
                                       uint32_t side, const int32_t *actions_host, int32_t *actions_dev,
                                       int spawn, int stable_max, int32_t *reward_dev, int32_t *reward_host,
                                       int8_t *obs_host, cgl_stream_t stream)
{
    return env_step_host_impl(win, wout, stable, n_envs, side, actions_host, actions_dev, spawn, stable_max,
                              reward_dev, reward_host, obs_host, stream, false);
}

extern "C" int cgl_stream_wait(cgl_stream_t stream)
{
    CGL_CUDA(cudaStreamSynchronize(as_stream(stream)));
    return 0;
}


// ---- IPC ------------------------------------------------------------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");

extern "C" int cgl_ipc_get_handle(void *dev_ptr, uint8_t handle_out[64])
{
    CGL_REQUIRE(dev_ptr && handle_out, CGL_E_BADARG, "cgl_ipc_get_handle: null");
    cudaIpcMemHandle_t h;
    CGL_CUDA(cudaIpcGetMemHandle(&h, dev_ptr));
    memcpy(handle_out, &h, 64);
    return 0;
}

extern "C" int cgl_ipc_open_handle(const uint8_t handle[64], void **dev_ptr_out)
{
    CGL_REQUIRE(handle && dev_ptr_out, CGL_E_BADARG, "cgl_ipc_open_handle: null");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CGL_CUDA(cudaIpcOpenMemHandle(dev_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}

extern "C" int cgl_ipc_close_handle(void *dev_ptr)
{
    CGL_REQUIRE(dev_ptr, CGL_E_BADARG, "cgl_ipc_close_handle: null");
    CGL_CUDA(cudaIpcCloseMemHandle(dev_ptr));
    return 0;
}

extern "C" int cgl_dev_alloc(uint64_t bytes, void **dev_ptr_out)
{
    CGL_REQUIRE(bytes && dev_ptr_out, CGL_E_BADARG, "cgl_dev_alloc: bad argument");
    CGL_CUDA(cudaMalloc(dev_ptr_out, bytes));
    CGL_CUDA(cudaMemset(*dev_ptr_out, 0, bytes));
    return 0;
}

extern "C" int cgl_dev_memset(void *dev_ptr, int value, uint64_t bytes, cgl_stream_t stream)
{
    CGL_REQUIRE(dev_ptr && bytes, CGL_E_BADARG, "cgl_dev_memset: bad argument");
    CGL_CUDA(cudaMemsetAsync(dev_ptr, value, bytes, as_stream(stream)));
    return 0;
}

extern "C" int cgl_dev_free(void *dev_ptr)
{
    CGL_CUDA(cudaFree(dev_ptr));
    return 0;
}

// ---- hardware-compressed device memory for the env state planes --------------------------------------------
// cuMemCreate with CU_MEM_ALLOCATION_COMP_GENERIC: the L2 compresses lines on their way to DRAM and expands them on
// the way back, so a stability plane that is mostly zero bytes moves fewer DRAM bytes per step while every kernel
// sees ordinary memory.  The driver API is reached through cudaGetDriverEntryPoint: the library links cudart
// statically and takes no libcuda dependency.
namespace {
struct DriverVmm {
    decltype(&::cuDeviceGetAttribute) dev_attr = nullptr;
    decltype(&::cuMemGetAllocationGranularity) granularity = nullptr;
    decltype(&::cuMemCreate) create = nullptr;
    decltype(&::cuMemGetAllocationPropertiesFromHandle) props = nullptr;
    decltype(&::cuMemAddressReserve) reserve = nullptr;
    decltype(&::cuMemMap) map = nullptr;
    decltype(&::cuMemSetAccess) access = nullptr;
    decltype(&::cuMemUnmap) unmap = nullptr;
    decltype(&::cuMemRelease) release = nullptr;
    decltype(&::cuMemAddressFree) address_free = nullptr;
    bool ok = false;
};

template <class F> bool entry(const char *name, F &fn)
{
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess ||
        !p) {
        cudaGetLastError();
        return false;
    }
    fn = reinterpret_cast<F>(p);
    return true;
}

const DriverVmm &vmm()
{
    static const DriverVmm d = [] {
        DriverVmm v;
        v.ok = entry("cuDeviceGetAttribute", v.dev_attr) && entry("cuMemGetAllocationGranularity", v.granularity) &&
               entry("cuMemCreate", v.create) && entry("cuMemGetAllocationPropertiesFromHandle", v.props) &&
               entry("cuMemAddressReserve", v.reserve) && entry("cuMemMap", v.map) &&
               entry("cuMemSetAccess", v.access) && entry("cuMemUnmap", v.unmap) &&
               entry("cuMemRelease", v.release) && entry("cuMemAddressFree", v.address_free);
        return v;
    }();
    return d;
}

CUmemAllocationProp compressible_prop(int device)
{
    CUmemAllocationProp p = {};
    p.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    p.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    p.location.id = device;
    p.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    return p;
}

// Allocation granularity of compressible memory on `device`; 0 if the device (or driver) does not offer it.
size_t compressible_granularity(int device)
{
    static size_t cached[64];
    static bool known[64] = {};
    if (device < 0 || device >= 64) return 0;
    if (known[device]) return cached[device];
    const DriverVmm &d = vmm();
    int supported = 0;
    size_t g = 0;
    if (d.ok && d.dev_attr(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, device) == CUDA_SUCCESS &&
        supported) {
        CUmemAllocationProp p = compressible_prop(device);
        if (d.granularity(&g, &p, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS) g = 0;
    }
    cached[device] = g;
    known[device] = true;
    return g;
}

// Every live allocation of cgl_state_alloc by base address: its size, and the physical handle if it is compressed
// (handle 0: the cudaMalloc fall-back).
struct StateBlock {
    size_t bytes;
    CUmemGenericAllocationHandle handle;
};
std::mutex g_state_mu;
std::map<uintptr_t, StateBlock> g_state_blocks;

void *compressed_alloc(size_t bytes, int device, CUmemGenericAllocationHandle *handle_out)
{
    const DriverVmm &d = vmm();
    const size_t g = compressible_granularity(device);
    if (!g) return nullptr;
    bytes = (bytes + g - 1) / g * g;
    CUmemAllocationProp p = compressible_prop(device);
    CUmemGenericAllocationHandle h = 0;
    if (d.create(&h, bytes, &p, 0) != CUDA_SUCCESS) return nullptr;
    CUmemAllocationProp got = {};
    if (d.props(&got, h) != CUDA_SUCCESS || got.allocFlags.compressionType != CU_MEM_ALLOCATION_COMP_GENERIC) {
        d.release(h);                              // not granted: the caller takes plain memory instead
        return nullptr;
    }
    CUdeviceptr va = 0;
    if (d.reserve(&va, bytes, g, 0, 0) != CUDA_SUCCESS) {
        d.release(h);
        return nullptr;
    }
    CUmemAccessDesc acc = {};
    acc.location = p.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (d.map(va, bytes, 0, h, 0) != CUDA_SUCCESS) {
        d.address_free(va, bytes);
        d.release(h);
        return nullptr;
    }
    if (d.access(va, bytes, &acc, 1) != CUDA_SUCCESS) {
        d.unmap(va, bytes);
        d.address_free(va, bytes);
        d.release(h);
        return nullptr;
    }
    *handle_out = h;
    return reinterpret_cast<void *>(va);
}
}  // namespace

extern "C" size_t cgl_state_granularity(int device) { return compressible_granularity(device); }

extern "C" void *cgl_state_alloc(size_t bytes, int device, cgl_stream_t)
{
    if (!bytes) return nullptr;
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) return nullptr;
    if (cur != device && cudaSetDevice(device) != cudaSuccess) return nullptr;
    CUmemGenericAllocationHandle h = 0;
    void *p = compressed_alloc(bytes, device, &h);
    if (p) {
        const size_t g = compressible_granularity(device);
        bytes = (bytes + g - 1) / g * g;
    } else if (cudaMalloc(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        p = nullptr;
    }
    if (cur != device) cudaSetDevice(cur);
    if (p) {
        std::lock_guard<std::mutex> lock(g_state_mu);
        g_state_blocks[reinterpret_cast<uintptr_t>(p)] = StateBlock{bytes, h};
    }
    return p;
}

extern "C" void cgl_state_free(void *ptr, size_t, int device, cgl_stream_t)
{
    if (!ptr) return;
    StateBlock b;
    {
        std::lock_guard<std::mutex> lock(g_state_mu);
        auto it = g_state_blocks.find(reinterpret_cast<uintptr_t>(ptr));
        if (it == g_state_blocks.end()) return;
        b = it->second;
        g_state_blocks.erase(it);
    }
    int cur = -1;
    cudaGetDevice(&cur);
    if (cur != device) cudaSetDevice(device);
    if (b.handle) {
        // cudaFree waits for the device; an unmap does not promise to, so wait here before the range goes away
        cudaDeviceSynchronize();
        const DriverVmm &d = vmm();
        const CUdeviceptr va = reinterpret_cast<CUdeviceptr>(ptr);
        d.unmap(va, b.bytes);
        d.release(b.handle);
        d.address_free(va, b.bytes);
    } else {
        cudaFree(ptr);
    }
    if (cur != device && cur >= 0) cudaSetDevice(cur);
}

extern "C" int cgl_state_compressed(const void *ptr)
{
    const uintptr_t a = reinterpret_cast<uintptr_t>(ptr);
    std::lock_guard<std::mutex> lock(g_state_mu);
    auto it = g_state_blocks.upper_bound(a);
    if (it == g_state_blocks.begin()) return 0;
    --it;
    return a < it->first + it->second.bytes && it->second.handle != 0;
}
