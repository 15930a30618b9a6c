// Host side of the launchers: the shared-memory budget, per-device kernel attributes, programmatic dependent
// launch and the A/B switches.  The state behind them lives in launch.cu; all of it is atomic or under a lock,
// so the first call on a device may come from any host thread.
#pragma once
#include <cstdlib>
#include <cuda_runtime.h>

namespace cube {

constexpr int kSmemPerBlock = 227 * 1024;    // dynamic shared memory of one block on sm_100a

// A/B switch (DESIGN.md 7b): `dflt` unless the value starts with the digit of the other state ('0' turns a
// default-on switch off, '1' a default-off switch on).  Call sites keep it in a function-local static const.
inline bool env_flag(const char* name, bool dflt)
{
    const char* e = getenv(name);
    return e && e[0] == (dflt ? '0' : '1') ? !dflt : dflt;
}

// integer switch: atoi of the value, `dflt` when unset; the call site checks the range
inline int env_int(const char* name, int dflt)
{
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

int sm_count();
// index of the current device for per-device launch state (cudaFuncSetAttribute is per device), 0..63
int device_slot();
// CTAs of a persistent (one-per-SM) grid: sm_count() minus the SMs the caller reserved for other
// kernels (cube_set_reserved_sms / CUBE_RESERVED_SMS), e.g. one for NCCL's reduction kernel
int persistent_ctas();
void set_reserved_sms(int n);
// grid of a persistent kernel: one CTA per `warps` tiles, at most persistent_ctas()
unsigned persistent_grid(long long n_tiles, int warps);

// warps whose buffers (`per_warp` bytes each, after `fixed` bytes) fit into kSmemPerBlock, at most `max_warps`
inline int warps_that_fit(int fixed, int per_warp, int max_warps)
{
    const int w = (kSmemPerBlock - fixed) / per_warp;
    return w < max_warps ? w : max_warps;
}

// Sets cudaFuncAttributeMaxDynamicSharedMemorySize of `kern` on the current device when `bytes` is more than
// was set there before (the limit only grows); returns the error of that call.
cudaError_t raise_smem_limit(const void* kern, int bytes);
// Sets the largest shared-memory carve-out of `kern` on the current device, once, so that occupancy is set by
// registers, not by the default split.  A hint: the result is ignored.
void prefer_max_shared(const void* kern);
template <typename F> cudaError_t raise_smem_limit(F* kern, int bytes) { return raise_smem_limit((const void*)kern, bytes); }
template <typename F> void prefer_max_shared(F* kern) { prefer_max_shared((const void*)kern); }

bool pdl_enabled();                          // CUBE_PDL

// Launch with programmatic stream serialisation (unless CUBE_PDL=0): the kernel may start while the previous
// kernel of the stream drains, and waits (griddepcontrol.wait) before its first global access.
template <typename... Params, typename... Args>
cudaError_t launch_pdl(void (*kern)(Params...), unsigned grid, unsigned block, int smem, cudaStream_t stream,
                       Args&&... args)
{
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = stream;
    cfg.attrs = &attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<Args&&>(args)...);
    return e != cudaSuccess ? e : cudaGetLastError();
}

}  // namespace cube
