// Host helpers of the C-ABI entry layer (lewin_abi.cu, lewin_conv.cu): the device query, the error return, pointer alignment
// and the workspace check.  Every entry decides its negative codes before its first launch, in this order: argument checks,
// workspace size and alignment (host arithmetic), then the device query.
#pragma once
#include "../../include/lewin_b200.h"
#include "ws_layout.h"

#include <cuda_runtime.h>
#include <stdint.h>

// return a failed cudaError_t (positive, as the header's error codes say)
#define CK(expr)                                            \
    do {                                                    \
        cudaError_t _e = (expr);                            \
        if (_e != cudaSuccess) return static_cast<int>(_e); \
    } while (0)

namespace lewin {

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
template <size_t N>
inline bool nonnull_aligned16(const void* const (&ps)[N]) {
    for (const void* p : ps)
        if (p && !aligned16(p)) return false;
    return true;
}

// The current device's SM count.  A failed runtime call returns its cudaError_t; a device that answers with a compute
// capability other than 10.x returns LEWIN_E_ARCH.
inline int device_sms(int* sms) {
    int dev = 0, cc = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&cc, cudaDevAttrComputeCapabilityMajor, dev);
    if (e != cudaSuccess) return static_cast<int>(e);
    return cc == 10 ? 0 : LEWIN_E_ARCH;
}

// Bytes of an entry's workspace: its layout function run in counting mode (per activation dtype where the layout has one).
template <typename Args, typename Ws>
size_t layout_bytes(Ws (*layout)(const Args*, WsLayout&), const Args* a) {
    WsLayout L;
    layout(a, L);
    return L.bytes;
}
template <typename Args, typename WsB, typename WsF>
size_t layout_bytes(int dtype, WsB (*bf16)(const Args*, WsLayout&), WsF (*f32)(const Args*, WsLayout&), const Args* a) {
    return dtype == LEWIN_DTYPE_BF16 ? layout_bytes(bf16, a) : layout_bytes(f32, a);
}

// An entry's steps after its argument checks: the workspace against its layout (none needed, or present, large enough and
// 16-byte aligned), the device query, then the layout carved from the workspace into `w` (L outlives w's slab registry).
template <typename Args, typename Ws>
int enter(void* ws, size_t ws_bytes, Ws (*layout)(const Args*, WsLayout&), const Args* a, WsLayout& L, Ws& w, int& sms) {
    const size_t need = layout_bytes(layout, a);
    if (need && (!ws || ws_bytes < need)) return LEWIN_E_WORKSPACE;
    if (need && !aligned16(ws)) return LEWIN_E_ALIGN;
    if (int rc = device_sms(&sms)) return rc;
    L.base = static_cast<unsigned char*>(ws);
    w = layout(a, L);
    return 0;
}

}  // namespace lewin
