// Loss side of the RL fine-tuning step (training.RLTrainer): clipped policy gradient, KL to a frozen teacher, entropy bonus and the
// value loss in normalised space, with their gradients wrt the head GEMM outputs, in one kernel (lib/action_head.py:176-220,
// lib/scaled_mse_head.py:37-43).  One CTA per frame row: the row's student (and teacher) log-probs of every head are staged in
// shared memory while the per-head KL / entropy sums are reduced, so every input byte is read from HBM once.
#pragma once
#include "common.cuh"

namespace vpt {

constexpr int kRlMaxHeads = 4;
constexpr int kRlThreads = 512;  // 3 CTAs (1536 threads) per SM: twice the loads in flight of 256

struct RlHeadsParams {
    const float* logp[kRlMaxHeads];    // student log-softmax [rows][n] per head
    const float* logp_t[kRlMaxHeads];  // teacher log-softmax (kTeacher only)
    const long long* idx[kRlMaxHeads]; // taken action per row
    int n[kRlMaxHeads], col0[kRlMaxHeads], soff[kRlMaxHeads];  // width, dlog column, shared-memory offset
    int nheads, ntot;
    const float *old_logp, *adv, *ret, *vpred, *mu_rsig;
    float clip_eps, kl_coef, ent_coef, vf_coef, inv_temp, inv_n;
    __nv_bfloat16* dlog;
    long long ld_out;
    int col_v;
    float* stats;  // [rows][5]: lp, kl, ent, (vpred - tn)^2, clipped
};

template <bool kTeacher>
__global__ void __launch_bounds__(kRlThreads) vpt_rl_heads_bwd_kernel(const RlHeadsParams p) {
    pdl_sync();
    extern __shared__ float s_row[];  // [ntot] student log-probs, then [ntot] teacher log-probs
    __shared__ float red[kRlThreads / 32][2 * kRlMaxHeads];
    __shared__ float tot[2 * kRlMaxHeads];
    __shared__ float s_g;
    const long long r = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float* s_lp = s_row;
    float* s_lt = s_row + p.ntot;

    // pass 1: stage the row, per-head sums of q (pd - pd_t) and -q pd
    float kl[kRlMaxHeads], ent[kRlMaxHeads];
#pragma unroll
    for (int h = 0; h < kRlMaxHeads; ++h) {
        kl[h] = 0.f;
        ent[h] = 0.f;
        if (h >= p.nheads) continue;
        const int n = p.n[h];
        const float* src = p.logp[h] + r * n;
        const float* srt = kTeacher ? p.logp_t[h] + r * n : nullptr;
        float* dl = s_lp + p.soff[h];
        float* dt = s_lt + p.soff[h];
        int j = tid;
        for (; j + 3 * kRlThreads < n; j += 4 * kRlThreads) {  // four loads in flight per thread
            float a[4], b[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) a[u] = __ldg(src + j + u * kRlThreads);
            if (kTeacher) {
#pragma unroll
                for (int u = 0; u < 4; ++u) b[u] = __ldg(srt + j + u * kRlThreads);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float q = __expf(a[u]);
                dl[j + u * kRlThreads] = a[u];
                ent[h] -= q * a[u];
                if (kTeacher) {
                    dt[j + u * kRlThreads] = b[u];
                    kl[h] += q * (a[u] - b[u]);
                }
            }
        }
        for (; j < n; j += kRlThreads) {
            const float a = __ldg(src + j);
            const float q = __expf(a);
            dl[j] = a;
            ent[h] -= q * a;
            if (kTeacher) {
                const float b = __ldg(srt + j);
                dt[j] = b;
                kl[h] += q * (a - b);
            }
        }
    }
#pragma unroll
    for (int h = 0; h < kRlMaxHeads; ++h) {
        kl[h] = warp_sum(kl[h]);
        ent[h] = warp_sum(ent[h]);
    }
    if (lane == 0) {
#pragma unroll
        for (int h = 0; h < kRlMaxHeads; ++h) {
            red[warp][2 * h] = kl[h];
            red[warp][2 * h + 1] = ent[h];
        }
    }
    __syncthreads();  // also publishes the staged row
    if (tid < 2 * kRlMaxHeads) {  // fixed-order sum over the warps
        float s = 0.f;
        for (int w = 0; w < kRlThreads / 32; ++w) s += red[w][tid];
        tot[tid] = s;
    }
    __syncthreads();

    // row coefficient of the policy-gradient term, value term, statistics
    if (tid == 0) {
        float lp = 0.f, klr = 0.f, entr = 0.f;
        for (int h = 0; h < p.nheads; ++h) {
            lp += s_lp[p.soff[h] + (int)__ldg(p.idx[h] + r)];
            klr += tot[2 * h];
            entr += tot[2 * h + 1];
        }
        const float A = __ldg(p.adv + r);
        const float ratio = __expf(lp - __ldg(p.old_logp + r));
        const bool clipped = (A > 0.f && ratio > 1.f + p.clip_eps) || (A < 0.f && ratio < 1.f - p.clip_eps);
        s_g = clipped ? 0.f : -ratio * A * p.inv_n;
        const float tn = (__ldg(p.ret + r) - __ldg(p.mu_rsig)) * __ldg(p.mu_rsig + 1);
        const float dv = __ldg(p.vpred + r) - tn;
        p.dlog[r * p.ld_out + p.col_v] = __float2bfloat16_rn(2.f * p.vf_coef * dv * p.inv_n);
        float* st = p.stats + r * 5;
        st[0] = lp;
        st[1] = klr;
        st[2] = entr;
        st[3] = dv * dv;
        st[4] = clipped ? 1.f : 0.f;
    }
    __syncthreads();
    const float g = s_g;
    const float kc = p.kl_coef * p.inv_n, ec = p.ent_coef * p.inv_n;

    // pass 2: d loss / d z = q (kc (pd - pd_t - kl_h) + ec (pd + H_h) - g) + g [j == a], times 1/temperature
    for (int h = 0; h < p.nheads; ++h) {
        const int n = p.n[h];
        const float* sl = s_lp + p.soff[h];
        const float* st = s_lt + p.soff[h];
        const float c = (kTeacher ? -kc * tot[2 * h] : 0.f) + ec * tot[2 * h + 1] - g;
        const int a = (int)__ldg(p.idx[h] + r);
        __nv_bfloat16* out = p.dlog + r * p.ld_out + p.col0[h];
        for (int j = tid; j < n; j += kRlThreads) {
            const float lpj = sl[j];
            const float q = __expf(lpj);
            float v = (kc + ec) * lpj + c;
            if (kTeacher) v -= kc * st[j];
            float gz = q * v;
            if (j == a) gz += g;
            out[j] = __float2bfloat16_rn(gz * p.inv_temp);
        }
    }
}

}  // namespace vpt

extern "C" int vpt_rl_heads_bwd(const float* const* logp, const float* const* logp_teacher, const int64_t* const* idx, const int32_t* n,
                                const int32_t* col0, int32_t nheads, const float* old_logp, const float* adv, const float* ret,
                                const float* vpred, const float* mu_rsig, float clip_eps, float kl_coef, float ent_coef, float vf_coef,
                                float inv_temp, float inv_n, void* dlog, int64_t ld_out, int32_t col_v, float* stats, int64_t rows,
                                void* stream) {
    using namespace vpt;
    VPT_CHECK(logp && idx && n && col0 && old_logp && adv && ret && vpred && mu_rsig && dlog && stats && rows > 0 && nheads >= 1 &&
                  nheads <= kRlMaxHeads && col_v >= 0 && col_v < ld_out,
              "vpt_rl_heads_bwd: bad arguments");
    RlHeadsParams p;
    memset(&p, 0, sizeof(p));
    int ntot = 0;
    for (int h = 0; h < nheads; ++h) {
        VPT_CHECK(logp[h] && idx[h] && (!logp_teacher || logp_teacher[h]) && n[h] > 0 && col0[h] >= 0 && (int64_t)col0[h] + n[h] <= ld_out &&
                      (col_v < col0[h] || col_v >= col0[h] + n[h]),
                  "vpt_rl_heads_bwd: bad head %d", h);
        p.logp[h] = logp[h];
        p.logp_t[h] = logp_teacher ? logp_teacher[h] : nullptr;
        p.idx[h] = reinterpret_cast<const long long*>(idx[h]);
        p.n[h] = n[h];
        p.col0[h] = col0[h];
        p.soff[h] = ntot;
        ntot += n[h];
    }
    const bool teacher = logp_teacher != nullptr;
    const size_t smem = (size_t)ntot * sizeof(float) * (teacher ? 2 : 1);
    VPT_CHECK(smem <= 200 * 1024, "vpt_rl_heads_bwd: %d head columns do not fit in shared memory", ntot);
    p.nheads = nheads;
    p.ntot = ntot;
    p.old_logp = old_logp;
    p.adv = adv;
    p.ret = ret;
    p.vpred = vpred;
    p.mu_rsig = mu_rsig;
    p.clip_eps = clip_eps;
    p.kl_coef = kl_coef;
    p.ent_coef = ent_coef;
    p.vf_coef = vf_coef;
    p.inv_temp = inv_temp;
    p.inv_n = inv_n;
    p.dlog = reinterpret_cast<__nv_bfloat16*>(dlog);
    p.ld_out = ld_out;
    p.col_v = col_v;
    p.stats = stats;
    if (teacher) {
        VPT_CUDA(cudaFuncSetAttribute(vpt_rl_heads_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        launch_k(vpt_rl_heads_bwd_kernel<true>, dim3((unsigned)rows), dim3(kRlThreads), smem, (cudaStream_t)stream, p);
    } else {
        VPT_CUDA(cudaFuncSetAttribute(vpt_rl_heads_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        launch_k(vpt_rl_heads_bwd_kernel<false>, dim3((unsigned)rows), dim3(kRlThreads), smem, (cudaStream_t)stream, p);
    }
    VPT_LAUNCH_CHECK();
    return VPT_OK;
}
