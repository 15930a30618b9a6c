// Host launch state (cube_launch.cuh): SM counts, reserved SMs, the counter slots of the dynamic tile
// scheduler (cube_sched.cuh) and the kernel attributes set so far.  Everything initialised lazily is atomic,
// a function-local static or under g_attr_lock, so the first call may come from any host thread.
#include <atomic>
#include <cstdint>
#include <mutex>
#include "cube_launch.cuh"
#include "cube_sched.cuh"

namespace sched {

__device__ Slot g_slots[kSlots];          // zero-initialised; every kernel re-arms its slot when it ends

Slot* claim_slot()
{
    static std::atomic<unsigned> seq{0};
    static std::atomic<Slot*> base[64];   // per device
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    Slot* b = base[dev].load(std::memory_order_relaxed);
    if (!b) {                             // threads that race here store the same address
        void* p = nullptr;
        if (cudaGetSymbolAddress(&p, g_slots) != cudaSuccess) return nullptr;
        b = static_cast<Slot*>(p);
        base[dev].store(b, std::memory_order_relaxed);
    }
    return b + (seq.fetch_add(1, std::memory_order_relaxed) % kSlots);
}

int tail_div()
{
    static const int v = [] {
        const int d = cube::env_int("CUBE_TAIL_DIV", kTailDiv);
        return d < 0 ? kTailDiv : d;
    }();
    return v;
}

}  // namespace sched

namespace cube {

namespace {

std::atomic<int> g_reserved_sms{-1};      // -1: CUBE_RESERVED_SMS not read yet

int reserved_sms()
{
    int v = g_reserved_sms.load(std::memory_order_relaxed);
    if (v < 0) {
        int env = env_int("CUBE_RESERVED_SMS", 0);
        if (env < 0) env = 0;
        // a value set by cube_set_reserved_sms before this first read wins over the environment
        if (g_reserved_sms.compare_exchange_strong(v, env, std::memory_order_relaxed)) v = env;
    }
    return v;
}

// Attributes set so far, per kernel (keyed by its address: instantiations of one template share a function
// type) and device.  An open-addressing table that only grows, and only under g_attr_lock: a launch whose
// kernel is configured already reads it without the lock.
struct KernelAttrs {
    std::atomic<const void*> kern;
    std::atomic<int> smem[64];                      // largest MaxDynamicSharedMemorySize set, 0 = none
    std::atomic<unsigned long long> carveout;       // devices the carve-out hint was set on, one bit each
};
constexpr size_t kKernels = 256;                    // ~50 kernels set attributes
KernelAttrs g_attrs[kKernels];
std::mutex g_attr_lock;                             // serialises the attribute calls and the inserts

// the entry of `kern`, or nullptr; with `add` (under g_attr_lock) a kernel without one gets a free entry
// (nullptr when the table is full: that kernel's attributes are then set on every call)
KernelAttrs* attrs_of(const void* kern, bool add)
{
    const size_t h = (reinterpret_cast<uintptr_t>(kern) >> 4) % kKernels;
    for (size_t i = 0; i < kKernels; ++i) {
        KernelAttrs& a = g_attrs[(h + i) % kKernels];
        const void* k = a.kern.load(std::memory_order_acquire);
        if (k == kern) return &a;
        if (!k) {
            if (!add) return nullptr;
            a.kern.store(kern, std::memory_order_release);
            return &a;
        }
    }
    return nullptr;
}

}  // namespace

int sm_count()
{
    static std::atomic<int> cached[64];   // per device, 0 = not asked yet (host threads may drive different devices)
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    std::atomic<int>& c = cached[dev & 63];
    int v = c.load(std::memory_order_relaxed);
    if (v == 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v < 1) v = 148;
        c.store(v, std::memory_order_relaxed);
    }
    return v;
}

int device_slot()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) dev = 0;
    return dev & 63;
}

int persistent_ctas()
{
    const int n = sm_count() - reserved_sms();
    return n < 1 ? 1 : n;
}

void set_reserved_sms(int n) { g_reserved_sms.store(n, std::memory_order_relaxed); }

unsigned persistent_grid(long long n_tiles, int warps)
{
    const long long grid = (n_tiles + warps - 1) / warps, cap = persistent_ctas();
    return (unsigned)(grid < cap ? grid : cap);
}

cudaError_t raise_smem_limit(const void* kern, int bytes)
{
    const int dev = device_slot();
    KernelAttrs* a = attrs_of(kern, false);
    if (a && bytes <= a->smem[dev].load(std::memory_order_acquire)) return cudaSuccess;
    std::lock_guard<std::mutex> lock(g_attr_lock);  // the limit only grows, whatever order threads get here in
    a = attrs_of(kern, true);
    if (a && bytes <= a->smem[dev].load(std::memory_order_relaxed)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess && a) a->smem[dev].store(bytes, std::memory_order_release);
    return e;
}

void prefer_max_shared(const void* kern)
{
    const unsigned long long bit = 1ull << device_slot();
    KernelAttrs* a = attrs_of(kern, false);
    if (a && (a->carveout.load(std::memory_order_acquire) & bit)) return;
    std::lock_guard<std::mutex> lock(g_attr_lock);
    a = attrs_of(kern, true);
    if (a && (a->carveout.load(std::memory_order_relaxed) & bit)) return;
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (a) a->carveout.fetch_or(bit, std::memory_order_release);
}

bool pdl_enabled()
{
    static const bool on = env_flag("CUBE_PDL", true);
    return on;
}

}  // namespace cube
