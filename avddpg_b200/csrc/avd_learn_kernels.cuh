// avd_learn_kernels.cuh -- host entry points of the tensor-core kernel families of the learn step: the persistent fused passes
// (avd_fused3.cu), the fused weight and data gradients (avd_wgrad3.cu, avd_dgrad3.cu) and the unfused GEMMs (avd_umma.cu).
#pragma once
#include <cuda_bf16.h>

#include <algorithm>

#include "avd_common.cuh"

namespace avd {

typedef __nv_bfloat16 bf16;

// Persistent CTAs per agent for R rows in 128-row tiles.  The dgrad and wgrad kernels each store one partial slice per CTA and
// unfold_kernel (avd_ddpg.cu) sums ctas_per_agent(A, R) of them, so every kernel family takes its grid from here.
inline int ctas_per_agent(int A, int64_t R) {
    const int tiles = (int)((R + 127) / 128);
    return std::max(1, std::min(tiles, sm_count() / std::max(1, A)));
}

namespace fused3 {

// The values are part of the kernels' mangled names (fused3_kernel<MODE, F16>), which profiling filters match.
// MODE_ACTOR_SAVE: the actor forward pass that also keeps what its backward needs -- sign bits of z1 (40 B per row) and of
// z2 + b2' (16 B), and d(action)/d(pre-activation) = high (1 - tanh^2) (4 B) -- so that the actor backward of the learn step is an
// elementwise kernel (actor_dm_kernel, avd_ddpg.cu).
enum Mode { MODE_ACTOR_OUT = 0, MODE_TARGET = 1, MODE_Q = 2, MODE_CRITIC_BWD = 3, MODE_CRITIC_ACTION = 5, MODE_ACTOR_SAVE = 6 };

// Arguments of one fused pass.  Fields a mode does not use stay at their defaults.
struct RunArgs {
    Mode mode = MODE_ACTOR_OUT;
    bool f16 = false;               // fp16 layer-2 operands (precision 2) instead of bf16
    avd_net_dims d = {};
    int A = 0;
    int64_t R = 0;
    const float* params = nullptr;  // [A][pstride]
    int64_t pstride = 0;
    const bf16* W2T = nullptr;      // 16-bit [A][128][F] folded layer-2 kernel, K-major (pack_fold_kernel / pack_fold4_kernel)
    const float* b2f = nullptr;     // [A][128] folded layer-2 bias
    const float* s = nullptr;       // element (n, k) at s[n*s_rs + k*s_cs]
    int64_t s_rs = 0, s_cs = 1;
    const float* act = nullptr;     // [A*R] critic passes
    const float* rew = nullptr;     // MODE_TARGET
    float gamma = 0.f, high = 0.f;
    const float* y = nullptr;       // MODE_CRITIC_BWD: TD targets
    const float* vtab = nullptr;    // MODE_CRITIC_ACTION: [A][vtab_floats()] from critic_vtab_kernel
    float* out = nullptr;           // forward modes: [A*R]; MODE_CRITIC_ACTION: d loss / d action; MODE_CRITIC_BWD: q (nullable)
    uint32_t* mask_out = nullptr;   // MODE_CRITIC_BWD / MODE_ACTOR_SAVE: [A*R][2*ceil(F/64)] sign masks of z1
    bf16* DZ_out = nullptr;         // MODE_CRITIC_BWD: 16-bit [A*R][128] = dm_scale * dq [z2 + b2' > 0]
    float dm_scale = 1.0f;
    float* sdq = nullptr;           // MODE_CRITIC_BWD: [A] += sum_n dq_n
    float* loss = nullptr;          // nullable; element 2*agent (+1 for the actor loss)
    uint32_t* mask2_out = nullptr;  // MODE_ACTOR_SAVE: [A*R][4] sign bits of z2 + b2'
    float* dact_out = nullptr;      // MODE_ACTOR_SAVE: [A*R] high (1 - tanh^2(pre-activation))
};

bool supported(const avd_net_dims& d);
int vtab_rows();
int vtab_stride();
int vtab_floats();
int run(const RunArgs& a, cudaStream_t st);

}  // namespace fused3

namespace wgrad3 {
// out: every CTA (agent, cta) stores its partial G2 (row-major [F][128] fp32, rows < F) at out + agent*out_agent_stride +
// cta*out_cta_stride.  DZ: 16-bit [A*R][128].
int run(bool f16, const avd_net_dims& d, bool critic, int A, int64_t R, const float* params, int64_t pstride, const float* s, int64_t s_rs,
        const float* act, const bf16* DZ, float* out, int64_t out_agent_stride, int64_t out_cta_stride, cudaStream_t st);
}

namespace dgrad3 {
int run(bool f16, int A, int64_t R, int F, const bf16* DZ, const bf16* W2b, const uint32_t* mask, int mask_words, const bf16* xextT, int64_t Rp,
        float* G1, int Fp, float* db2, int64_t db2_stride, cudaStream_t st);
}

namespace umma {
// bf16 GEMM, layout 0 = TN (C = A B^T), 1 = NT (C += A^T B, split-K).  planes = 1: plain bf16 operands; planes = 3: hi / mid / lo
// planes, plane p of batch b at A + (p * batch + b) * a_batch (avd_gemm_bf16x3).
int gemm_bf16(int planes, int layout, int batch, int M, int N, int K, const void* A, int64_t lda, int64_t a_batch, const void* B, int64_t ldb,
              int64_t b_batch, float* C, int64_t ldc, int64_t c_batch, int splitk, cudaStream_t st);
}

}  // namespace avd
