// libvpt_b200.so -- single translation unit (unity build) of the sm_100a kernels behind include/vpt_b200.h.
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC vpt_b200.cu -o libvpt_b200.so
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include "common.cuh"

namespace vpt {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
}  // namespace vpt

#include "gemm_tc.cuh"
#include "wgrad_tc.cuh"
#include "gemv_small.cuh"
#include "conv_zp.cuh"
#include "conv_zp_t.cuh"
#include "elementwise.cuh"
#include "firstconv.cuh"
#include "conv3d.cuh"
#include "attention.cuh"
#include "heads.cuh"
#include "adam.cuh"
#include "resize.cuh"
#include "backward.cuh"
#include "attention_bwd.cuh"
#include "firstconv_bwd.cuh"
#include "precise.cuh"
#include "codec.cuh"
#include "rl_heads.cuh"

extern "C" const char* vpt_last_error(void) { return vpt::g_err; }
extern "C" int vpt_abi_version(void) { return VPT_ABI_VERSION; }
extern "C" int vpt_num_sms(void) { return vpt::num_sms(); }
extern "C" int vpt_set_pdl(int32_t on) {
    vpt::g_pdl = on ? 1 : 0;
    return VPT_OK;
}
extern "C" int vpt_device_error(void) {
    unsigned int v = 0;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        vpt::set_error("cudaDeviceSynchronize: %s", cudaGetErrorString(e));
        return VPT_ERR_CUDA;
    }
    e = cudaMemcpyFromSymbol(&v, vpt::g_device_error, sizeof(v));
    if (e != cudaSuccess) {
        vpt::set_error("cudaMemcpyFromSymbol: %s", cudaGetErrorString(e));
        return VPT_ERR_CUDA;
    }
    if (v != 0) {
        unsigned int z = 0;
        cudaMemcpyToSymbol(vpt::g_device_error, &z, sizeof(z));
        vpt::set_error("device watchdog: mbarrier wait timed out (code 0x%x)", v);
        return VPT_ERR_DEVICE;
    }
    return VPT_OK;
}
