// Host-side helpers shared by the C-ABI translation units: error reporting, TMA descriptor
// construction through the driver entry point (no link-time libcuda dependency), launch counting.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>
#include <string>
#include <utility>

namespace pk {

void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;
int sm_count();

// Encode a tiled bf16 tensor map (rank 2..5), 128B swizzle, zero OOB fill.
//   dims[0] is the contiguous dimension; strides_bytes[i] is the stride of dims[i+1].
bool make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box);

// Programmatic dependent launch.  Kernels that execute pdl_launch_dependents() + pdl_wait() (common.cuh) before their
// first global-memory access are launched with the programmatic-stream-serialization attribute: the next such kernel
// in the stream is scheduled while this one drains, runs its prologue (barrier init, TMEM allocation, descriptor
// prefetch) on the SMs that have gone idle and blocks in griddepcontrol.wait until this grid has completed and its
// writes are visible - stream semantics are unchanged, the launch gap and the prologue leave the critical path.
// pk_set_pdl(0) / PK_PDL=0 turn the attribute off (the device-side wait is then a no-op).
bool pdl_enabled();
int set_pdl(int on);
struct PdlLaunch {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[2];
  PdlLaunch(dim3 grid, dim3 block, size_t smem, cudaStream_t st, unsigned cluster_x = 0) {
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    unsigned n = 0;
    if (cluster_x > 1) {
      attr[n].id = cudaLaunchAttributeClusterDimension;
      attr[n].val.clusterDim.x = cluster_x;
      attr[n].val.clusterDim.y = 1;
      attr[n].val.clusterDim.z = 1;
      ++n;
    }
    if (pdl_enabled()) {
      attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[n].val.programmaticStreamSerializationAllowed = 1;
      ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
  }
};
// launch a kernel that begins with pdl_launch_dependents() / pdl_wait()
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
  PdlLaunch L(grid, block, smem, st);
  return cudaLaunchKernelEx(&L.cfg, kernel, std::forward<Args>(args)...);
}

// Tile of the decoder's implicit-GEMM 3x3 convolution: `pixels` pixels as TW = min(W, 64) columns x TH rows, which
// must divide the W x H image (pixels = 128 for the forward / dgrad, 64 for the wgrad).  Every entry point that
// handles the conv output checks it, so that all of them accept the same image sizes.
inline bool conv_tile_geometry(int H, int W, int pixels, int* TW, int* TH) {
  const int tw = W < 64 ? W : 64;
  if (tw <= 0 || W % tw != 0 || pixels % tw != 0) return false;
  const int th = pixels / tw;
  if (H <= 0 || H % th != 0) return false;
  *TW = tw;
  *TH = th;
  return true;
}

#define PK_CHECK(cond, ...)      \
  do {                           \
    if (!(cond)) {               \
      pk::set_error(__VA_ARGS__); \
      return 1;                  \
    }                            \
  } while (0)

#define PK_LAUNCH_CHECK(name)                                                        \
  do {                                                                               \
    cudaError_t e__ = cudaGetLastError();                                            \
    if (e__ != cudaSuccess) {                                                        \
      pk::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));         \
      return 2;                                                                      \
    }                                                                                \
    pk::g_launches.fetch_add(1, std::memory_order_relaxed);                          \
  } while (0)

}  // namespace pk
