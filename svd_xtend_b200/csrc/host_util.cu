#include "host_util.h"
#include "../../include/svd_xtend_b200.h"
#include <stdio.h>

static thread_local char g_err[512] = "";

int svdx_fail(int code, const char* msg) {
  snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}
int svdx_fail_cuda(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return SVDX_E_CUDA;
}
extern "C" const char* svdx_last_error(void) { return g_err; }

int svdx_device_slot(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) return 0;
  return dev < SVDX_MAX_DEVICES ? dev : SVDX_MAX_DEVICES - 1;
}

extern "C" int svdx_num_sms(void) {
  static int n[SVDX_MAX_DEVICES] = {0};
  const int slot = svdx_device_slot();
  if (n[slot] == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) return 148;
    n[slot] = v;
  }
  return n[slot];
}

// kernels of the CURRENT device may dereference memory of `peer_device` (its allocations, or another process's allocations on
// it mapped here through CUDA IPC) once peer access is enabled on the current device's context; idempotent
extern "C" int svdx_enable_peer_access(int32_t peer_device) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return svdx_fail_cuda(e, "enable_peer_access: cudaGetDevice");
  if (dev == peer_device) return SVDX_OK;
  int can = 0;
  e = cudaDeviceCanAccessPeer(&can, dev, peer_device);
  if (e != cudaSuccess) return svdx_fail_cuda(e, "enable_peer_access: cudaDeviceCanAccessPeer");
  if (!can) return svdx_fail(SVDX_E_BADARG, "enable_peer_access: the two GPUs are not peer-capable (no NVLink / PCIe P2P path)");
  e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return SVDX_OK; }
  if (e != cudaSuccess) return svdx_fail_cuda(e, "enable_peer_access: cudaDeviceEnablePeerAccess");
  return SVDX_OK;
}

// ---- CUDA IPC of a device buffer between the ranks of one node (one process per GPU): the owner exports the handle of the
// allocation that contains `ptr` plus ptr's byte offset inside it; a consumer opens it WITH ITS OWN DEVICE CURRENT, so the
// mapping is made for (and peer access lazily enabled from) the GPU whose kernels will dereference it.
typedef CUresult (*AddrRangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);
extern "C" int svdx_ipc_export(const void* ptr, void* handle_out, int64_t* offset_out) {
  if (!ptr || !handle_out || !offset_out) return svdx_fail(SVDX_E_BADARG, "ipc_export: null argument");
  static AddrRangeFn range = nullptr;
  if (!range) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess) return svdx_fail(SVDX_E_NODRIVER, "ipc_export: cuMemGetAddressRange unavailable");
    range = reinterpret_cast<AddrRangeFn>(p);
  }
  CUdeviceptr base = 0;
  size_t size = 0;
  if (range(&base, &size, reinterpret_cast<CUdeviceptr>(ptr)) != CUDA_SUCCESS) return svdx_fail(SVDX_E_BADARG, "ipc_export: not a device allocation");
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, reinterpret_cast<void*>(base));
  if (e != cudaSuccess) return svdx_fail_cuda(e, "ipc_export: cudaIpcGetMemHandle");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  memcpy(handle_out, &h, 64);
  *offset_out = (int64_t)(reinterpret_cast<CUdeviceptr>(ptr) - base);
  return SVDX_OK;
}
extern "C" int svdx_ipc_import(const void* handle, int64_t offset, void** ptr_out) {
  if (!handle || !ptr_out || offset < 0) return svdx_fail(SVDX_E_BADARG, "ipc_import: bad argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  void* base = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return svdx_fail_cuda(e, "ipc_import: cudaIpcOpenMemHandle");
  *ptr_out = static_cast<char*>(base) + offset;
  return SVDX_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int svdx_make_tmap_ex(CUtensorMap* out, const void* base, int f32, int swizzle_bytes, int rank, const uint64_t* dims,
                      const uint64_t* strides, const uint32_t* box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return svdx_fail(SVDX_E_NODRIVER, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bx[5];
  cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides[i];
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                              : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                              : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(out, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank,
                   const_cast<void*>(base), gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[256];
    snprintf(buf, sizeof(buf), "cuTensorMapEncodeTiled failed (%d): rank %d dims %llu %llu %llu box %u %u %u stride0 %llu", (int)r,
             rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
             (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0,
             (unsigned long long)(rank > 1 ? strides[0] : 0));
    return svdx_fail(SVDX_E_CUDA, buf);
  }
  return 0;
}

int svdx_make_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides,
                   const uint32_t* box) {
  return svdx_make_tmap_ex(out, base, 0, 128, rank, dims, strides, box);
}

extern "C" int svdx_struct_size(int which) {
  return which == 0 ? (int)sizeof(SvdxTapGemm) : which == 1 ? (int)sizeof(SvdxAttn) : which == 2 ? (int)sizeof(SvdxClipPixels) : -1;
}
