// avd_ddpg.cu -- DDPG learn step for a population of agents (workers/trainer.py:472-508 + 345-356).
//
// Data flow (all launches batched over the A agents; rows of agent a are [a*R, (a+1)*R)):
//   target actor(s')  -> a'      | layer1 -> GEMM(l1 x l2)      -> head(tanh)
//   target critic(s',a') -> y    | layer1 -> GEMM((l1+la) x l2) -> head(+TD target r + gamma q')
//   critic(s,a) -> q, dLc/dz2    | layer1 -> GEMM -> head-backward (MSE grad, head/BN/bias grads, dz2)
//                                | wgrad GEMM (cat^T dz2), dgrad GEMM (dz2 W2^T), layer1-backward
//   actor(s) -> pi ; critic(s,pi)| layer1 -> GEMM -> head ; layer1 -> GEMM -> head-backward(action only)
//                                | dgrad (action columns) -> d pi ; actor head-backward, wgrad, dgrad, layer1-backward
//   Adam x2 (TF-Keras form), Polyak x2
// The three big contractions (forward, wgrad, dgrad on the l1 x l2 and (l1+la) x l2 layers, 97% of the FLOPs)
// go through `gemm_batched`, which dispatches on io->precision: 0 = fp32 SIMT tiles (parity mode, this
// file), 1 = bf16 tcgen05/TMEM tensor-core kernels, 2 = the same kernels with fp16 layer-2 operands (11-bit significand;
// the backward tile stays bf16) and the T formulation of the critic-action pass (avd_fused3.cu), 3 = the unfused tcgen05 GEMMs on
// three-way split bf16 operands (umma::gemm_bf16 on hi / mid / lo planes, fp32-accurate).  Everything else (K=ns and K=1 layers,
// heads with N=1, BatchNorm affine, reductions for bias/BN gradients, TD target, losses) is fused into the
// layer1 / head kernels below.
//
// BatchNormalization is always the inference affine (models are never called with training=True):
//   y = g*(x-mu)/sqrt(var+1e-3)+be, with trainable g/be and frozen mu/var (SURVEY.md §3.3).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "avd_common.cuh"
#include "avd_ddpg_layout.cuh"
#include "avd_learn_kernels.cuh"
#include "avd_umma.cuh"

namespace avd {

// GEMM operand written as three bf16 planes (precision 3): element i is hi at p[i], mid at p[plane + i], lo at p[2 plane + i],
// hi = bf16(x), mid = bf16(x - hi), lo = bf16(x - hi - mid).  Both differences are exact in fp32, so hi + mid + lo keeps 24 bits of x.
// Behaves like an output pointer (offset, null test) so that the producers take it in place of float* / bf16*.
struct Planes3 {
    bf16* p;
    int64_t plane;
    __host__ __device__ Planes3 operator+(int64_t i) const { return Planes3{p + i, plane}; }
    __host__ __device__ explicit operator bool() const { return p != nullptr; }
};

// Format of the GEMM operands of the unfused learn step and forward passes (H, H1a, DZ and the W2 packs), set by the precision:
// fp32 (0), one bf16 copy (1 and 2) or three bf16 planes (3).  A bf16 copy is given as much workspace as fp32.
enum OperandFormat { OPND_F32, OPND_BF16, OPND_BF16X3 };
inline OperandFormat operand_format(int precision) { return precision == 0 ? OPND_F32 : precision == 3 ? OPND_BF16X3 : OPND_BF16; }
inline int operand_planes(int precision) { return operand_format(precision) == OPND_BF16X3 ? 3 : 1; }
inline int64_t operand_bytes(int precision, int64_t n) {     // workspace of an operand of n elements
    return operand_format(precision) == OPND_BF16X3 ? n * 3 * (int64_t)sizeof(bf16) : n * (int64_t)sizeof(float);
}

// The operand at p as T: float*, bf16* or Planes3 (plane = elements per plane)
template <typename T> __host__ __device__ __forceinline__ T as_operand(void* p, int64_t) { return reinterpret_cast<T>(p); }
template <> __host__ __device__ __forceinline__ Planes3 as_operand<Planes3>(void* p, int64_t plane) { return Planes3{reinterpret_cast<bf16*>(p), plane}; }

// Calls f with the operand at p typed by the precision's format; f picks the kernel instantiation from the argument's type
template <class Fn>
void with_operand(int precision, void* p, int64_t plane, Fn&& f) {
    switch (operand_format(precision)) {
        case OPND_F32: f(as_operand<float*>(p, plane)); break;
        case OPND_BF16: f(as_operand<bf16*>(p, plane)); break;
        case OPND_BF16X3: f(as_operand<Planes3>(p, plane)); break;
    }
}

__device__ __forceinline__ void split3(float x, bf16& hi, bf16& mid, bf16& lo) {
    hi = __float2bfloat16_rn(x);
    const float r = x - __bfloat162float(hi);
    mid = __float2bfloat16_rn(r);
    lo = __float2bfloat16_rn(r - __bfloat162float(mid));
}

__device__ __forceinline__ void store_out(float* p, float v) { *p = v; }
__device__ __forceinline__ void store_out(bf16* p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void store_out(Planes3 o, float v) {
    bf16 h, m, l;
    split3(v, h, m, l);
    o.p[0] = h;
    o.p[o.plane] = m;
    o.p[2 * o.plane] = l;
}

// ------------------------------------------------------------------------------------------------
// layer 1: H[n][f] = bn(relu(x[n] . W[:,f] + b[f]))   (state columns, then -- critic -- action columns)
// ------------------------------------------------------------------------------------------------
constexpr int kL1Rows = 128;
constexpr int kL1BwdRows = 256;

__device__ __forceinline__ void store_pair(float* p, float v0, float v1) { *reinterpret_cast<float2*>(p) = make_float2(v0, v1); }
__device__ __forceinline__ void store_pair(bf16* p, float v0, float v1) {
    *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(v0, v1);
}
__device__ __forceinline__ void store_pair(Planes3 o, float v0, float v1) {
    bf16 h0, m0, l0, h1, m1, l1;
    split3(v0, h0, m0, l0);
    split3(v1, h1, m1, l1);
    *reinterpret_cast<__nv_bfloat162*>(o.p) = __halves2bfloat162(h0, h1);
    *reinterpret_cast<__nv_bfloat162*>(o.p + o.plane) = __halves2bfloat162(m0, m1);
    *reinterpret_cast<__nv_bfloat162*>(o.p + 2 * o.plane) = __halves2bfloat162(l0, l1);
}

// One thread owns a PAIR of adjacent columns (packed 4/8-byte stores, a warp writes 128/256 contiguous bytes per row);
// l1 and la must be even so that a pair never straddles the state/action boundary.  TOut: float*, bf16* or Planes3.
template <bool CRITIC, typename TOut>
__global__ void __launch_bounds__(128) l1_forward_kernel(avd_net_dims d, const float* __restrict__ params, int64_t pstride,
                                                         const float* __restrict__ s, int64_t s_rs, int64_t s_cs,
                                                         const float* __restrict__ act, int64_t R, TOut H) {
    const int agent = blockIdx.y;
    const float* P = params + (int64_t)agent * pstride;
    const int F = CRITIC ? d.l1 + d.la : d.l1;
    const int64_t row0 = (int64_t)blockIdx.x * kL1Rows;
    const int nrows = (int)min((int64_t)kL1Rows, R - row0);
    const int64_t base = (int64_t)agent * R + row0;
    const int nx = d.ns + (CRITIC ? 1 : 0);
    __shared__ float xs[kL1Rows][9];  // up to 8 state words + action
    for (int i = threadIdx.x; i < nrows * nx; i += blockDim.x) {
        const int r = i / nx, k = i % nx;
        xs[r][k] = (k < d.ns) ? s[(base + r) * s_rs + k * s_cs] : act[base + r];
    }
    __syncthreads();
    for (int f = 2 * threadIdx.x; f < F; f += 2 * blockDim.x) {
        const bool is_act = CRITIC && f >= d.l1;
        const int c = is_act ? f - d.l1 : f;
        int64_t oW, ob, og, obe, omu, ovar;
        if (CRITIC) {
            const CriticOff o = critic_off(d);
            oW = is_act ? o.Wa : o.Ws; ob = is_act ? o.ba : o.bs; og = is_act ? o.ga : o.gs; obe = is_act ? o.bea : o.bes;
            omu = is_act ? o.mua : o.mus; ovar = is_act ? o.vara : o.vars;
        } else {
            const ActorOff o = actor_off(d);
            oW = o.W1; ob = o.b1; og = o.g1; obe = o.be1; omu = o.mu1; ovar = o.var1;
        }
        const int width = is_act ? d.la : d.l1;
        const int nin = is_act ? 1 : d.ns;
        const int xoff = is_act ? d.ns : 0;
        float w0[8], w1[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            w0[k] = (k < nin) ? P[oW + (int64_t)k * width + c] : 0.0f;
            w1[k] = (k < nin) ? P[oW + (int64_t)k * width + c + 1] : 0.0f;
        }
        const float b0 = P[ob + c], b1 = P[ob + c + 1];
        const float inv0 = 1.0f / sqrtf(P[ovar + c] + kBnEps), inv1 = 1.0f / sqrtf(P[ovar + c + 1] + kBnEps);
        const float sc0 = P[og + c] * inv0, sc1 = P[og + c + 1] * inv1;
        const float sh0 = P[obe + c] - P[omu + c] * sc0, sh1 = P[obe + c + 1] - P[omu + c + 1] * sc1;
        for (int r = 0; r < nrows; ++r) {
            float z0 = b0, z1 = b1;
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (k < nin) {
                    const float x = xs[r][xoff + k];
                    z0 = fmaf(x, w0[k], z0);
                    z1 = fmaf(x, w1[k], z1);
                }
            store_pair(H + (base + r) * F + f, fmaf(fmaxf(z0, 0.0f), sc0, sh0), fmaf(fmaxf(z1, 0.0f), sc1, sh1));
        }
    }
}

// layer-1 backward: from dH[n][f] accumulate dW, db, dg, dbe (one set of atomics per CTA and column).
// The kernel is instruction-issue bound (ncu: 73 % issue-active), so the inner loop is kept minimal: inputs of a
// row come from ONE 16-byte shared-memory broadcast, rows past the end are zero-padded instead of clamped, and the
// state / action columns run in separately specialised loops.
template <bool CRITIC>
__global__ void __launch_bounds__(128) l1_backward_kernel(avd_net_dims d, const float* __restrict__ params, int64_t pstride,
                                                          const float* __restrict__ s, int64_t s_rs, const float* __restrict__ act, int64_t R,
                                                          const float* __restrict__ dH, float* __restrict__ grads, int64_t gstride) {
    constexpr int ROWS = kL1BwdRows;
    const int agent = blockIdx.y;
    const float* P = params + (int64_t)agent * pstride;
    float* G = grads + (int64_t)agent * gstride;
    const int F = CRITIC ? d.l1 + d.la : d.l1;
    const int64_t row0 = (int64_t)blockIdx.x * ROWS;
    const int nrows = (int)min((int64_t)ROWS, R - row0);
    const int64_t base = (int64_t)agent * R + row0;
    __shared__ float4 xs4[ROWS];     // state words 0..3 (ns <= 4 fast path; words 4..7 in xs_hi)
    __shared__ float4 xs_hi[ROWS];
    __shared__ float xa[ROWS];
    for (int r = threadIdx.x; r < ROWS; r += blockDim.x) {
        float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (r < nrows)
            for (int k = 0; k < d.ns; ++k) v[k] = s[(base + r) * s_rs + k];
        xs4[r] = make_float4(v[0], v[1], v[2], v[3]);
        xs_hi[r] = make_float4(v[4], v[5], v[6], v[7]);
        xa[r] = (CRITIC && r < nrows) ? act[base + r] : 0.0f;
    }
    __syncthreads();
    const int nrows8 = (nrows + 7) & ~7;
    // ---- state columns
    {
        int64_t oW, ob, og, obe, omu, ovar;
        if (CRITIC) { const CriticOff o = critic_off(d); oW = o.Ws; ob = o.bs; og = o.gs; obe = o.bes; omu = o.mus; ovar = o.vars; }
        else { const ActorOff o = actor_off(d); oW = o.W1; ob = o.b1; og = o.g1; obe = o.be1; omu = o.mu1; ovar = o.var1; }
        for (int f = threadIdx.x; f < d.l1; f += blockDim.x) {
            float w[8], dw[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) { w[k] = (k < d.ns) ? P[oW + (int64_t)k * d.l1 + f] : 0.0f; dw[k] = 0.0f; }
            const float b = P[ob + f], mu = P[omu + f];
            const float inv = 1.0f / sqrtf(P[ovar + f] + kBnEps);
            const float ginv = P[og + f] * inv;
            float db = 0.0f, dg = 0.0f, dbe = 0.0f;
            const float* dcol = dH + base * F + f;
            for (int r0 = 0; r0 < nrows8; r0 += 8) {
                float dhv[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) dhv[u] = (r0 + u < nrows) ? dcol[(int64_t)(r0 + u) * F] : 0.0f;   // 8 loads in flight
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float4 x = xs4[r0 + u];
                    float z = fmaf(x.x, w[0], fmaf(x.y, w[1], fmaf(x.z, w[2], fmaf(x.w, w[3], b))));
                    float4 xh4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (d.ns > 4) {
                        xh4 = xs_hi[r0 + u];
                        z = fmaf(xh4.x, w[4], fmaf(xh4.y, w[5], fmaf(xh4.z, w[6], fmaf(xh4.w, w[7], z))));
                    }
                    const float dh = dhv[u];
                    dg = fmaf(dh, (fmaxf(z, 0.0f) - mu) * inv, dg);
                    dbe += dh;
                    const float dz = z > 0.0f ? dh * ginv : 0.0f;
                    db += dz;
                    dw[0] = fmaf(x.x, dz, dw[0]); dw[1] = fmaf(x.y, dz, dw[1]); dw[2] = fmaf(x.z, dz, dw[2]); dw[3] = fmaf(x.w, dz, dw[3]);
                    if (d.ns > 4) {
                        dw[4] = fmaf(xh4.x, dz, dw[4]); dw[5] = fmaf(xh4.y, dz, dw[5]); dw[6] = fmaf(xh4.z, dz, dw[6]); dw[7] = fmaf(xh4.w, dz, dw[7]);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (k < d.ns) atomicAdd(G + oW + (int64_t)k * d.l1 + f, dw[k]);
            atomicAdd(G + ob + f, db);
            atomicAdd(G + og + f, dg);
            atomicAdd(G + obe + f, dbe);
        }
    }
    // ---- action columns (critic only)
    if (CRITIC) {
        const CriticOff o = critic_off(d);
        for (int c = threadIdx.x; c < d.la; c += blockDim.x) {
            const float w = P[o.Wa + c], b = P[o.ba + c], mu = P[o.mua + c];
            const float inv = 1.0f / sqrtf(P[o.vara + c] + kBnEps);
            const float ginv = P[o.ga + c] * inv;
            float dw = 0.0f, db = 0.0f, dg = 0.0f, dbe = 0.0f;
            const float* dcol = dH + base * F + d.l1 + c;
            for (int r0 = 0; r0 < nrows8; r0 += 8) {
                float dhv[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) dhv[u] = (r0 + u < nrows) ? dcol[(int64_t)(r0 + u) * F] : 0.0f;
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float a = xa[r0 + u];
                    const float z = fmaf(a, w, b);
                    const float dh = dhv[u];
                    dg = fmaf(dh, (fmaxf(z, 0.0f) - mu) * inv, dg);
                    dbe += dh;
                    const float dz = z > 0.0f ? dh * ginv : 0.0f;
                    db += dz;
                    dw = fmaf(a, dz, dw);
                }
            }
            atomicAdd(G + o.Wa + c, dw);
            atomicAdd(G + o.ba + c, db);
            atomicAdd(G + o.ga + c, dg);
            atomicAdd(G + o.bea + c, dbe);
        }
    }
}

// d(action)[n] = sum_f dza[n][f] * Wa[f], dza = dHa * ga*inva * (za > 0): the critic -> actor link (trainer.py:503-506)
// One thread per row; the la (<= 64) per-column parameters are staged in shared memory.
__global__ void __launch_bounds__(256) action_grad_kernel(avd_net_dims d, const float* __restrict__ params, int64_t pstride,
                                                          const float* __restrict__ act, int64_t R, const float* __restrict__ dHa,
                                                          float* __restrict__ dact) {
    const CriticOff o = critic_off(d);
    const int agent = blockIdx.y;
    const float* P = params + (int64_t)agent * pstride;
    __shared__ float wa[64], ba[64], gi[64];
    for (int f = threadIdx.x; f < d.la; f += blockDim.x) {
        wa[f] = P[o.Wa + f];
        ba[f] = P[o.ba + f];
        gi[f] = P[o.ga + f] / sqrtf(P[o.vara + f] + kBnEps);
    }
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = (int64_t)agent * R + r;
        const float a = act[n];
        const float4* row = reinterpret_cast<const float4*>(dHa + n * d.la);
        float acc = 0.0f;
        for (int f4 = 0; f4 < d.la / 4; ++f4) {
            const float4 v = row[f4];
            const float dv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int f = 4 * f4 + j;
                const float z = fmaf(a, wa[f], ba[f]);
                acc = fmaf(z > 0.0f ? dv[j] * gi[f] : 0.0f, wa[f], acc);
            }
        }
        dact[n] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// heads: everything after the l2-wide GEMM.  One warp per row, lane owns columns lane, lane+32, ...
// ------------------------------------------------------------------------------------------------
// HEAD_CRITIC_TARGET_HP: the TD target with every agent's own gamma (HeadArgs.hp); a mode of its own so that HEAD_CRITIC_TARGET
// compiles to the kernel it was before.
enum HeadMode { HEAD_ACTOR_FWD = 0, HEAD_CRITIC_TARGET = 1, HEAD_CRITIC_Q = 2, HEAD_CRITIC_BWD = 3, HEAD_CRITIC_BWD_ACTION = 4, HEAD_ACTOR_BWD = 5,
                HEAD_CRITIC_TARGET_HP = 6 };

struct HeadArgs {
    const float* params;   // [A][pstride]
    int64_t pstride;
    int64_t o_b2, o_g2, o_be2, o_mu2, o_var2, o_W3, o_b3;
    const float* Z;        // [A*R][L2] raw GEMM output (bias not yet added)
    int64_t R;
    float high, gamma;
    const float* hp;       // TARGET_HP: [A][4] per-agent (gamma, ...); gamma of agent a = hp[4 a] instead of `gamma`
    const float* rew;      // TARGET
    const float* y;        // CRITIC_BWD
    const float* dpi;      // ACTOR_BWD
    float* out;            // ACTOR_FWD: action, TARGET: y, Q/BWD: q (nullable for BWD)
    void* DZ;              // BWD modes: float* (precision 0), bf16* (precision 1 / 2) or three bf16 planes (precision 3)
    int64_t dz_plane;      // precision 3: elements per plane of DZ (all agents' rows)
    float* grads;          // [A][gstride] (BWD, ACTOR_BWD)
    int64_t gstride;
    float* loss;           // [A][2] nullable
};

template <int MODE, int CPL, typename TDZ>   // CPL = columns per lane (l2 = 32*CPL); TDZ: float*, bf16* or Planes3
__global__ void __launch_bounds__(256) head_kernel(HeadArgs h) {
    constexpr int L2 = 32 * CPL;
    constexpr int ROWS = 64;
    constexpr bool BWD = MODE == HEAD_CRITIC_BWD || MODE == HEAD_ACTOR_BWD;
    const int agent = blockIdx.y;
    const float* P = h.params + (int64_t)agent * h.pstride;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t row0 = (int64_t)blockIdx.x * ROWS;
    const int nrows = (int)min((int64_t)ROWS, h.R - row0);
    float b2[CPL], sc[CPL], sh[CPL], inv[CPL], mu[CPL], w3[CPL], ginv[CPL];
    float aW3[CPL], aG[CPL], aBe[CPL], aB2[CPL];
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
        const int c = lane + 32 * j;
        b2[j] = P[h.o_b2 + c];
        inv[j] = 1.0f / sqrtf(P[h.o_var2 + c] + kBnEps);
        mu[j] = P[h.o_mu2 + c];
        ginv[j] = P[h.o_g2 + c] * inv[j];
        sc[j] = ginv[j];
        sh[j] = P[h.o_be2 + c] - mu[j] * sc[j];
        w3[j] = P[h.o_W3 + c];
        aW3[j] = aG[j] = aBe[j] = aB2[j] = 0.0f;
    }
    const float b3 = P[h.o_b3];
    const float invR = 1.0f / (float)h.R;
    float aB3 = 0.0f, aLoss = 0.0f;
    for (int r = wid; r < nrows; r += 8) {
        const int64_t n = (int64_t)agent * h.R + row0 + r;
        float z[CPL], hh[CPL];
        float part = 0.0f;
#pragma unroll
        for (int j = 0; j < CPL; ++j) {
            z[j] = h.Z[n * L2 + lane + 32 * j] + b2[j];
            hh[j] = fmaf(fmaxf(z[j], 0.0f), sc[j], sh[j]);
            part = fmaf(hh[j], w3[j], part);
        }
        const float pre = warp_sum(part) + b3;
        if (MODE == HEAD_ACTOR_FWD) {
            if (lane == 0) h.out[n] = h.high * tanhf(pre);
        } else if (MODE == HEAD_CRITIC_TARGET || MODE == HEAD_CRITIC_TARGET_HP) {
            const float gamma = MODE == HEAD_CRITIC_TARGET_HP ? h.hp[4 * agent] : h.gamma;
            if (lane == 0) h.out[n] = h.rew[n] + gamma * pre;      // trainer.py:494 (no terminal mask)
        } else if (MODE == HEAD_CRITIC_Q) {
            if (lane == 0) h.out[n] = pre;
        } else {
            float dq;
            if (MODE == HEAD_CRITIC_BWD) {
                const float diff = pre - h.y[n];
                dq = 2.0f * diff * invR;                           // d mean((y-q)^2) / dq
                aLoss = fmaf(diff, diff * invR, aLoss);
                if (h.out && lane == 0) h.out[n] = pre;
            } else if (MODE == HEAD_CRITIC_BWD_ACTION) {
                dq = -invR;                                        // d(-mean(q)) / dq
                aLoss -= pre * invR;
            } else {  // HEAD_ACTOR_BWD
                const float t = tanhf(pre);
                dq = h.dpi[n] * h.high * (1.0f - t * t);
            }
            if (BWD) aB3 += dq;
#pragma unroll
            for (int j = 0; j < CPL; ++j) {
                const float dh = dq * w3[j];
                const float dz = z[j] > 0.0f ? dh * ginv[j] : 0.0f;
                store_out(as_operand<TDZ>(h.DZ, h.dz_plane) + n * L2 + lane + 32 * j, dz);
                if (BWD) {
                    aW3[j] = fmaf(hh[j], dq, aW3[j]);
                    aG[j] = fmaf(dh, (fmaxf(z[j], 0.0f) - mu[j]) * inv[j], aG[j]);
                    aBe[j] += dh;
                    aB2[j] += dz;
                }
            }
        }
    }
    if (MODE == HEAD_CRITIC_BWD || MODE == HEAD_CRITIC_BWD_ACTION || MODE == HEAD_ACTOR_BWD) {
        __shared__ float red[8][L2];
        __shared__ float red1[8][2];
        float* G = BWD ? h.grads + (int64_t)agent * h.gstride : nullptr;
        if (BWD) {
            const int64_t offs[4] = {h.o_W3, h.o_g2, h.o_be2, h.o_b2};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
#pragma unroll
                for (int j = 0; j < CPL; ++j) red[wid][lane + 32 * j] = (q == 0 ? aW3[j] : q == 1 ? aG[j] : q == 2 ? aBe[j] : aB2[j]);
                __syncthreads();
                if (threadIdx.x < L2) {
                    float s = 0.0f;
#pragma unroll
                    for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
                    atomicAdd(G + offs[q] + threadIdx.x, s);
                }
                __syncthreads();
            }
        }
        if (lane == 0) { red1[wid][0] = aB3; red1[wid][1] = aLoss; }   // lane 0 holds the row-level sums (all lanes equal)
        __syncthreads();
        if (threadIdx.x == 0) {
            float sb = 0.0f, sl = 0.0f;
            for (int w = 0; w < 8; ++w) { sb += red1[w][0]; sl += red1[w][1]; }
            if (BWD) atomicAdd(G + h.o_b3, sb);
            if (h.loss && MODE != HEAD_ACTOR_BWD) atomicAdd(h.loss + 2 * agent + (MODE == HEAD_CRITIC_BWD ? 0 : 1), sl);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// fp32 SIMT GEMM, strided + batched: C[b] (MxN) (+)= A[b] (MxK) B[b] (KxN).  64x64x16 tiles, 4x4 per thread.
// ------------------------------------------------------------------------------------------------
struct GemmArgs {
    const float* A; int64_t a_m, a_k, a_batch;   // element (m,k) at A[b*a_batch + m*a_m + k*a_k]
    const float* B; int64_t b_k, b_n, b_batch;
    float* C; int64_t c_m, c_n, c_batch;
    int M, N, K, splitk;
};

template <bool A_KCONTIG, bool B_NCONTIG>
__global__ void __launch_bounds__(256) sgemm_kernel(GemmArgs g) {
    constexpr int BM = 64, BN = 64, BK = 16;
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int batch = blockIdx.z / g.splitk, split = blockIdx.z % g.splitk;
    const float* A = g.A + (int64_t)batch * g.a_batch;
    const float* B = g.B + (int64_t)batch * g.b_batch;
    float* C = g.C + (int64_t)batch * g.c_batch;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int kchunk = (((g.K + g.splitk - 1) / g.splitk) + BK - 1) / BK * BK;
    const int kbeg = split * kchunk, kend = min(g.K, kbeg + kchunk);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4] = {};
    for (int k0 = kbeg; k0 < kend; k0 += BK) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = threadIdx.x + i * 256;
            int m, k;
            if (A_KCONTIG) { k = e & 15; m = e >> 4; } else { m = e & 63; k = e >> 6; }
            const int gm = m0 + m, gk = k0 + k;
            As[k][m] = (gm < g.M && gk < kend) ? A[(int64_t)gm * g.a_m + (int64_t)gk * g.a_k] : 0.0f;
            int n, kb;
            if (B_NCONTIG) { n = e & 63; kb = e >> 6; } else { kb = e & 15; n = e >> 4; }
            const int gn = n0 + n, gkb = k0 + kb;
            Bs[kb][n] = (gn < g.N && gkb < kend) ? B[(int64_t)gkb * g.b_k + (int64_t)gn * g.b_n] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= g.M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= g.N) continue;
            float* dst = C + (int64_t)gm * g.c_m + (int64_t)gn * g.c_n;
            if (g.splitk > 1) atomicAdd(dst, acc[i][j]); else *dst = acc[i][j];
        }
    }
}

static int launch_sgemm(const GemmArgs& g, int nbatch, cudaStream_t st) {
    dim3 grid((g.N + 63) / 64, (g.M + 63) / 64, nbatch * g.splitk);
    const bool ak = g.a_k == 1, bn = g.b_n == 1;
    if (ak && bn) sgemm_kernel<true, true><<<grid, 256, 0, st>>>(g);
    else if (ak && !bn) sgemm_kernel<true, false><<<grid, 256, 0, st>>>(g);
    else if (!ak && bn) sgemm_kernel<false, true><<<grid, 256, 0, st>>>(g);
    else sgemm_kernel<false, false><<<grid, 256, 0, st>>>(g);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

// ------------------------------------------------------------------------------------------------
// optimiser, targets, federated reductions
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ params, int64_t pstride, const float* __restrict__ grads,
                                                   int64_t gstride, float* __restrict__ m, float* __restrict__ v,
                                                   const int32_t* __restrict__ step, const uint8_t* __restrict__ mask, int64_t n,
                                                   float lr, float b1, float b2, float eps) {
    const int agent = blockIdx.y;
    if (mask && !mask[agent]) return;
    const float t = (float)(step[agent] + 1);
    const float lr_t = lr * sqrtf(1.0f - powf(b2, t)) / (1.0f - powf(b1, t));
    float* P = params + (int64_t)agent * pstride;
    const float* G = grads + (int64_t)agent * gstride;
    float* Mm = m + (int64_t)agent * n;
    float* Vv = v + (int64_t)agent * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float g = G[i];
        const float mi = Mm[i] + (g - Mm[i]) * (1.0f - b1);
        const float vi = Vv[i] + (g * g - Vv[i]) * (1.0f - b2);
        Mm[i] = mi;
        Vv[i] = vi;
        P[i] -= lr_t * mi / (sqrtf(vi) + eps);
    }
}

// Actor and critic in one launch (blockIdx.z): the two updates are independent and each is only a few microseconds long.
struct AdamNet {
    float *params, *target;
    const float* grads;
    float *m, *v;
    const int32_t* step;
    int64_t pstride, gstride, n_train, total;
    float lr;
};
struct AdamNets { AdamNet n[2]; };

// HP: per-agent learning rates and tau from hp[A][4] = (gamma, actor_lr, critic_lr, tau) (avd_learn_io.agent_hp), same arithmetic; a
// template parameter so that the launch without a table compiles to the kernel it was before.
template <bool HP>
__global__ void __launch_bounds__(256) adam_polyak2_kernel(AdamNets nets, const uint8_t* __restrict__ mask, float b1, float b2, float eps, float tau,
                                                           const float* __restrict__ hp) {
    pdl_wait();                  // launched with programmatic dependent launch (avd_common.cuh): every CTA waits before it reads or exits
    pdl_launch_dependents();
    const AdamNet& nt = nets.n[blockIdx.z];
    const int agent = blockIdx.y;
    if (mask && !mask[agent]) return;
    const float lr = HP ? hp[4 * agent + (blockIdx.z == 0 ? 2 : 1)] : nt.lr;      // n[0] is the critic
    if (HP) tau = hp[4 * agent + 3];
    const float t = (float)(nt.step[agent] + 1);
    const float lr_t = lr * sqrtf(1.0f - powf(b2, t)) / (1.0f - powf(b1, t));
    float* P = nt.params + (int64_t)agent * nt.pstride;
    float* T = nt.target + (int64_t)agent * nt.pstride;
    const float* G = nt.grads + (int64_t)agent * nt.gstride;
    float* Mm = nt.m + (int64_t)agent * nt.n_train;
    float* Vv = nt.v + (int64_t)agent * nt.n_train;
    const float omt = 1.0f - tau;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nt.total; i += (int64_t)gridDim.x * blockDim.x) {
        float p = P[i];
        if (i < nt.n_train) {
            const float g = G[i];
            const float mi = Mm[i] + (g - Mm[i]) * (1.0f - b1);
            const float vi = Vv[i] + (g * g - Vv[i]) * (1.0f - b2);
            Mm[i] = mi;
            Vv[i] = vi;
            p -= lr_t * mi / (sqrtf(vi) + eps);
            P[i] = p;
        }
        T[i] = p * tau + T[i] * omt;
    }
}

__global__ void step_increment2_kernel(int32_t* step_a, int32_t* step_b, const uint8_t* mask, int A) {
    pdl_wait();
    pdl_launch_dependents();
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a < A && (!mask || mask[a])) {
        step_a[a] += 1;
        step_b[a] += 1;
    }
}

__global__ void step_increment_kernel(int32_t* step, const uint8_t* mask, int A) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a < A && (!mask || mask[a])) step[a] += 1;
}

__global__ void __launch_bounds__(256) polyak_kernel(float* __restrict__ target, const float* __restrict__ online,
                                                     const uint8_t* __restrict__ mask, int64_t n, float tau) {
    const int agent = blockIdx.y;
    if (mask && !mask[agent]) return;
    float* T = target + (int64_t)agent * n;
    const float* O = online + (int64_t)agent * n;
    const float omt = 1.0f - tau;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        T[i] = O[i] * tau + T[i] * omt;   // ddpgagent.py:46,53: variable * tau + target * (1 - tau)
}

__global__ void __launch_bounds__(256) fed_reduce_kernel(float* __restrict__ out, int64_t out_pitch, const float* __restrict__ in,
                                                         int64_t pitch, int n_members, int64_t stride_s, int64_t stride_x,
                                                         const float* __restrict__ weights, const float* __restrict__ scale, int64_t n) {
    const int s = blockIdx.y;
    const float sc = scale ? scale[s] : 1.0f / (float)n_members;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float acc = 0.0f;
        for (int x = 0; x < n_members; ++x) {
            const float w = weights ? weights[(int64_t)s * n_members + x] : 1.0f;
            acc = fmaf(w, in[((int64_t)s * stride_s + (int64_t)x * stride_x) * pitch + i], acc);
        }
        out[(int64_t)s * out_pitch + i] = sc * acc;
    }
}

// Both banks of a federated round in one launch: out[s][0..na) / out[s][na..na+nc) = sum_x w[s][x] * actor / critic vector of
// member (s, x), and the divisor column out[s][na+nc] = sum_x w[s][x] (or the member count) that turns the exchanged sums into
// the mean (federated.py:62) or the weighted mean (federated.py:110).
__global__ void __launch_bounds__(256) fed_reduce2_kernel(float* __restrict__ out, int64_t out_pitch, const float* __restrict__ in_a,
                                                          int64_t pitch_a, int64_t na, const float* __restrict__ in_c, int64_t pitch_c,
                                                          int64_t nc, int n_members, int64_t stride_s, int64_t stride_x,
                                                          const float* __restrict__ weights) {
    const int s = blockIdx.y;
    const int64_t n = na + nc;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += (int64_t)gridDim.x * blockDim.x) {
        float acc = 0.0f;
        if (i == n) {
            for (int x = 0; x < n_members; ++x) acc += weights ? weights[(int64_t)s * n_members + x] : 1.0f;
        } else {
            const float* in = i < na ? in_a : in_c;
            const int64_t pitch = i < na ? pitch_a : pitch_c, col = i < na ? i : i - na;
            for (int x = 0; x < n_members; ++x) {
                const float w = weights ? weights[(int64_t)s * n_members + x] : 1.0f;
                acc = fmaf(w, in[((int64_t)s * stride_s + (int64_t)x * stride_x) * pitch + col], acc);
            }
        }
        out[(int64_t)s * out_pitch + i] = acc;
    }
}

// ... and the way back: member (s, x) of both banks receives columns [0, na) / [na, na+nc) of system s (set_weights, trainer.py:448-456)
__global__ void __launch_bounds__(256) fed_broadcast2_kernel(float* __restrict__ out_a, int64_t pitch_a, int64_t na, float* __restrict__ out_c,
                                                             int64_t pitch_c, int64_t nc, const float* __restrict__ in, int64_t in_pitch,
                                                             int n_members, int64_t stride_s, int64_t stride_x, const uint8_t* __restrict__ mask) {
    const int s = blockIdx.y, x = blockIdx.z;
    const int64_t member = (int64_t)s * stride_s + (int64_t)x * stride_x;
    if (mask && !mask[member]) return;
    const int64_t n = na + nc;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = in[(int64_t)s * in_pitch + i];
        if (i < na) out_a[member * pitch_a + i] = v;
        else out_c[member * pitch_c + (i - na)] = v;
    }
}

// Trainer.get_weight (workers/trainer.py:385-398) for every agent at once: |1 / mean(last `window` episodic rewards)|, the episodic
// reward of agent (g, m) being the mean over its group's E platoons.  One CTA per agent; ep_hist is the ring the env kernel keeps.
__global__ void __launch_bounds__(256) fed_weights_kernel(const float* __restrict__ ep_hist, int window, int M, int64_t G, int64_t E,
                                                          float* __restrict__ out, int transpose) {
    const int m = blockIdx.x / (int)G;
    const int64_t g = blockIdx.x - (int64_t)m * G;
    const int64_t P = G * E;
    float acc = 0.0f;
    for (int64_t i = threadIdx.x; i < (int64_t)window * E; i += blockDim.x) {
        const int64_t k = i / E, e = i - k * E;
        acc += ep_hist[(k * M + m) * P + g * E + e];
    }
    __shared__ float red[8];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += red[k];
        const float mean = t / (float)((int64_t)window * E);
        out[transpose ? g * M + m : (int64_t)m * G + g] = fabsf(1.0f / mean);
    }
}

__global__ void __launch_bounds__(256) fed_finalize_kernel(float* __restrict__ buf, int64_t pitch, int64_t n) {
    float* row = buf + (int64_t)blockIdx.y * pitch;
    const float inv = 1.0f / row[n];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) row[i] *= inv;
}

__global__ void __launch_bounds__(256) fed_broadcast_kernel(float* __restrict__ out, int64_t out_pitch, const float* __restrict__ in,
                                                            int64_t in_pitch, int n_members, int64_t stride_s, int64_t stride_x,
                                                            const uint8_t* __restrict__ mask, int64_t n) {
    const int s = blockIdx.y, x = blockIdx.z;
    const int64_t member = (int64_t)s * stride_s + (int64_t)x * stride_x;
    if (mask && !mask[member]) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[member * out_pitch + i] = in[(int64_t)s * in_pitch + i];
}

// ------------------------------------------------------------------------------------------------
// bf16 copies of the layer-2 kernels for the tensor-core path: W2b [F][l2] (dgrad B operand, K-major) and
// W2T [l2][F] (forward B operand, K-major); TOut = bf16* (precision 1 / 2) or Planes3 (precision 3)
// ------------------------------------------------------------------------------------------------
template <typename TOut>
__global__ void __launch_bounds__(256) pack_w2_kernel(const float* __restrict__ params, int64_t pstride, int64_t oW2, int F, int l2,
                                                      TOut W2b, TOut W2T) {
    const int agent = blockIdx.y;
    const float* W = params + (int64_t)agent * pstride + oW2;
    const int n = F * l2;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int f = i / l2, c = i - f * l2;
        const float v = W[i];
        if (W2b) store_out(W2b + ((int64_t)agent * n + i), v);
        store_out(W2T + ((int64_t)agent * n + (int64_t)c * F + f), v);
    }
}

// 16-bit operand element: bf16 (precision 1) or fp16 (precision 2); both travel as bf16-typed pointers (TMA moves raw 16-bit words)
__device__ __forceinline__ bf16 to_op16(float v, int f16) {
    if (f16) {       // saturating, like the F2FP.SATFINITE conversions of the kernels: never inf from a finite value
        const __half h = __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f));
        return *reinterpret_cast<const bf16*>(&h);
    }
    return __float2bfloat16_rn(v);
}
__device__ __forceinline__ float round_op16(float v, int f16) {
    return f16 ? __half2float(__float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f))) : __bfloat162float(__float2bfloat16_rn(v));
}

// BN-folded packing for the fused tensor-core path.  With h1 = r1*sc1 + sh1 (r1 = relu(z1), inference BatchNorm):
//   z2 = h1 W2 + b2 = r1 W2' + b2',   W2'[f][j] = sc1[f] W2[f][j],   b2'[j] = b2[j] + sum_f sh1[f] W2[f][j]
// W2T [l2][F] is the forward B operand (K-major), W2b [F][l2] the dgrad B operand (nullable), b2f [l2] fp32.
// One CTA per agent and 32-column slab of l2; thread (fy, j) walks features fy, fy+8, ...
struct FoldOff {
    int64_t W2, b2;
    int64_t g[2], be[2], mu[2], var[2];   // BN of the state columns [0] and of the action columns [1]
    int l1;                               // features < l1 use set 0
};

// b2'[j] = b2[j] + sum_f sh1[f] W2[f][j] of one agent in a fixed order: warp fy sums features fy, fy + 8, ..., then warp 0 adds
// the eight partial sums in warp order.  Called by all 256 threads of the CTAs of feature slab 0 only: adding per-slab partial sums
// with atomics made b2', and with it every output of the pass, depend on the order in which CTAs finished (the same weights at two
// agent slots, or in two calls, gave outputs a few ulp apart).  These CTAs are the tail of the launch, so sh1 is computed once per
// feature into shared memory and every W2 load of a thread is issued before the first is used.  F <= kFoldMaxF: the fused path
// (fused3::supported) has F = 256 + la <= 304.
constexpr int kFoldMaxF = 320;
__device__ __forceinline__ void fold_bias(const float* __restrict__ P, const FoldOff& o, int F, int l2, int j, int fy, float* __restrict__ b2f) {
    __shared__ float red[8][32];
    __shared__ float sh_s[kFoldMaxF];
    for (int f = threadIdx.x; f < F; f += blockDim.x) {
        const bool st = f < o.l1;
        const int c = st ? f : f - o.l1;
        const float sc = P[(st ? o.g[0] : o.g[1]) + c] / sqrtf(P[(st ? o.var[0] : o.var[1]) + c] + kBnEps);
        sh_s[f] = P[(st ? o.be[0] : o.be[1]) + c] - P[(st ? o.mu[0] : o.mu[1]) + c] * sc;
    }
    float w[kFoldMaxF / 8];
#pragma unroll
    for (int k = 0; k < kFoldMaxF / 8; ++k) {
        const int f = fy + 8 * k;
        w[k] = (j < l2 && f < F) ? P[o.W2 + (int64_t)f * l2 + j] : 0.0f;
    }
    __syncthreads();
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < kFoldMaxF / 8; ++k) {
        const int f = fy + 8 * k;
        if (f < F) acc += sh_s[f] * w[k];
    }
    red[fy][threadIdx.x & 31] = acc;
    __syncthreads();
    if (fy == 0 && j < l2) {
        float t = P[o.b2 + j];
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
        *b2f = t;
    }
}

__global__ void __launch_bounds__(256) pack_fold_kernel(const float* __restrict__ params, int64_t pstride, FoldOff o, int F, int l2,
                                                        bf16* __restrict__ W2b, bf16* __restrict__ W2T, float* __restrict__ b2f, int f16) {
    // grid: (l2/32 column slabs, feature slabs of 8, agents); thread (fy, j) owns feature blockIdx.y*8 + fy, column j.
    // The CTAs of the first feature slab also write b2f (fold_bias).
    const int agent = blockIdx.z;
    const float* P = params + (int64_t)agent * pstride;
    const int j = blockIdx.x * 32 + (threadIdx.x & 31);
    const int fy = threadIdx.x >> 5;
    const int f = blockIdx.y * 8 + fy;
    if (j < l2 && f < F) {
        const bool st = f < o.l1;
        const int c = st ? f : f - o.l1;
        const float sc = P[(st ? o.g[0] : o.g[1]) + c] / sqrtf(P[(st ? o.var[0] : o.var[1]) + c] + kBnEps);
        const float w = P[o.W2 + (int64_t)f * l2 + j];
        const bf16 v = to_op16(sc * w, f16);
        if (W2b) W2b[((int64_t)agent * F + f) * l2 + j] = v;
        W2T[((int64_t)agent * l2 + j) * F + f] = v;
    }
    if (blockIdx.y == 0) fold_bias(P, o, F, l2, j, fy, b2f + (int64_t)agent * l2 + j);
}

// The four networks of a learn step (target actor, target critic, critic, actor) in ONE launch: blockIdx.z = job * A + agent.
struct FoldJob {
    const float* params;
    int64_t pstride;
    FoldOff o;
    int64_t g2, var2, W3;       // head: BatchNorm 2 scale / variance and the output weights (for w3' = sc2 w3)
    int F;
    bf16 *W2b, *W2T;            // W2b (dgrad operand, nullable): [F][l2] = W2' diag(w3');  W2T (forward operand): [l2][F] = W2'^T
    float* b2f;
    float* wscale;              // fp16 only, nullable: [A] 1 / s.  W2b is scaled by s = 2^-e, max_j |w3'_j| 2^-e in [0.5, 1):
                                // the products W2' w3' (~1e-5 at initialisation) would otherwise sit in the subnormal range of fp16
};
constexpr int kFoldJobs = 4;
struct FoldJobs { FoldJob j[kFoldJobs]; };

__device__ __forceinline__ void pack_fold4_body(const FoldJobs& jobs, int A, int l2, int f16, int bx, int by, int bz) {
    const int job = bz / A, agent = bz - job * A;
    const FoldJob& jb = jobs.j[job];
    if (by * 8 >= jb.F) return;
    float s_w3 = 1.0f;          // the power-of-two scale s of this (net, agent): every CTA derives it from the same 128 head weights
    if (f16 && jb.W2b) {
        __shared__ float mx[8];
        const float* Pq = jb.params + (int64_t)agent * jb.pstride;
        float m = 0.0f;
        for (int jj = threadIdx.x; jj < l2; jj += blockDim.x) m = fmaxf(m, fabsf(Pq[jb.W3 + jj] * Pq[jb.g2 + jj] / sqrtf(Pq[jb.var2 + jj] + kBnEps)));
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o2));
        if ((threadIdx.x & 31) == 0) mx[threadIdx.x >> 5] = m;
        __syncthreads();
        m = mx[0];
#pragma unroll
        for (int k = 1; k < 8; ++k) m = fmaxf(m, mx[k]);
        if (m > 0.0f && m < 3.0e38f) {
            int e;
            frexpf(m, &e);
            e = max(-100, min(100, e));
            s_w3 = ldexpf(1.0f, -e);
        }
        if (jb.wscale && bx == 0 && by == 0 && threadIdx.x == 0) jb.wscale[agent] = 1.0f / s_w3;
        __syncthreads();
    }
    const FoldOff& o = jb.o;
    const float* P = jb.params + (int64_t)agent * jb.pstride;
    const int F = jb.F;
    const int j = bx * 32 + (threadIdx.x & 31);
    const int fy = threadIdx.x >> 5;
    const int f = by * 8 + fy;
    if (j < l2 && f < F) {
        const bool st = f < o.l1;
        const int c = st ? f : f - o.l1;
        const float sc = P[(st ? o.g[0] : o.g[1]) + c] / sqrtf(P[(st ? o.var[0] : o.var[1]) + c] + kBnEps);
        const float w = P[o.W2 + (int64_t)f * l2 + j];
        // the backward tile carries dq [z2 > 0] without the head weight (avd_fused3.cu): dR = dm (W2' diag(w3'))^T
        if (jb.W2b) {
            const float w3p = P[jb.W3 + j] * P[jb.g2 + j] / sqrtf(P[jb.var2 + j] + kBnEps) * s_w3;
            jb.W2b[((int64_t)agent * F + f) * l2 + j] = to_op16(sc * w * w3p, f16);
        }
        jb.W2T[((int64_t)agent * l2 + j) * F + f] = to_op16(sc * w, f16);
    }
    if (by == 0) fold_bias(P, o, F, l2, j, fy, jb.b2f + (int64_t)agent * l2 + j);
}

// xextT[agent][c][r] (bf16, row pitch Rp): x_ext = [ s_hi(4) a_hi 1 0 0 | s_lo(4) a_lo 0 0 0 ] of row r, stored transposed so that a
// [16][128-row] tile is the K-major B operand of the fused dgrad kernel (avd_dgrad3.cu):
//   G1[f][c] = sum_n dz1[n][f] x_ext[n][c]  =>  dW1[k][f] = G1[f][k] + G1[f][8+k],  dWa[f] = G1[l1+f][4] + G1[l1+f][12],  db[f] = G1[f][5]
// and column 5 (the constant one) also yields db2 = sum_n dz2[n][:].
__device__ __forceinline__ void xext_body(const float* __restrict__ s, int64_t s_rs, const float* __restrict__ a, int ns, int64_t N,
                                          bf16* __restrict__ xextT, int64_t R, int64_t Rp, int f16, int64_t block) {
    const int64_t n = block * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float v[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < ns && k < 4; ++k) v[k] = s[n * s_rs + k];
    v[4] = a[n];
    bf16 hi[8], lo[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { hi[k] = to_op16(0.0f, f16); lo[k] = hi[k]; }
#pragma unroll
    for (int k = 0; k < 5; ++k) {       // hi/lo split in the operand format of the dgrad kernel (bf16: 16 bits of v, fp16: 22)
        hi[k] = to_op16(v[k], f16);
        lo[k] = to_op16(v[k] - round_op16(v[k], f16), f16);
    }
    hi[5] = to_op16(1.0f, f16);
    const int64_t agent = n / R, r = n - agent * R;
    bf16* col = xextT + agent * 16 * Rp + r;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        col[(int64_t)k * Rp] = hi[k];
        col[(int64_t)(8 + k) * Rp] = lo[k];
    }
}

// V table of the critic-action pass (avd_fused3.cu, MODE_CRITIC_ACTION): the action reaches the critic through one scalar, so
// d q / d a = sum_j [z2_j + b2'_j > 0] V[k(a)][j] with V[k][j] = sum_{f active in interval k} wa_f W2'[l1 + f][j] w3'_j, k(a) = number of
// breakpoints -ba_f / wa_f below a.  Grid (agents, 4 column slabs of 32); 256 threads = 32 columns x 8 row groups.  Every CTA sorts
// the breakpoints (rank sort, la <= 64), stages its [la][32] slab of wa_f W2' w3' in shared memory with coalesced loads, and fills
// its rows -- the active set of interval k is evaluated with the forward pass's own test fma(a, wa_f, ba_f) > 0 at a point inside
// the interval.  Output per agent: [rows][stride] fp32 (pad columns zero) followed by 64 sorted breakpoints (+inf padded).
__device__ __forceinline__ void critic_vtab_body(const float* __restrict__ params, int64_t pstride, const CriticOff& o, const avd_net_dims& d,
                                                 float* __restrict__ vtab, int rows, int stride, int total, int agent, int slab) {
    const int tid = threadIdx.x;
    const float* P = params + (int64_t)agent * pstride;
    float* out = vtab + (int64_t)agent * total;
    __shared__ float wa[64], ba[64], brk[64], sorted[64], col[64][33];
    const int la = d.la;
    const float inf = __int_as_float(0x7f800000);
    if (tid < 64) {
        const float w = tid < la ? P[o.Wa + tid] : 0.0f, b = tid < la ? P[o.ba + tid] : 0.0f;
        wa[tid] = w;
        ba[tid] = b;
        brk[tid] = (tid < la && w != 0.0f) ? -b / w : inf;
        sorted[tid] = inf;
    }
    for (int i = tid; i < 64 * 32; i += blockDim.x) {        // col[f][c] = wa_f sc_a,f W2[l1 + f][j] w3'_j,  j = 32 slab + c
        const int f = i >> 5, c = i & 31, jj = slab * 32 + c;
        float v = 0.0f;
        if (f < la && jj < d.l2) {
            const float sca = P[o.ga + f] / sqrtf(P[o.vara + f] + kBnEps);
            const float w3p = P[o.W3 + jj] * P[o.g2 + jj] / sqrtf(P[o.var2 + jj] + kBnEps);
            v = P[o.Wa + f] * sca * P[o.W2 + (int64_t)(d.l1 + f) * d.l2 + jj] * w3p;
        }
        col[f][c] = v;
    }
    __syncthreads();
    if (tid < la) {       // rank sort (ties broken by index)
        const float t = brk[tid];
        int rank = 0;
        for (int g2 = 0; g2 < la; ++g2) rank += (brk[g2] < t || (brk[g2] == t && g2 < tid)) ? 1 : 0;
        sorted[rank] = t;
    }
    __syncthreads();
    int m = 0;          // finite breakpoints
    for (int i = 0; i < la; ++i) m += sorted[i] < inf ? 1 : 0;
    if (slab == 0) {
        if (tid < 64) out[rows * stride + tid] = sorted[tid];
        for (int i = rows * stride + 64 + tid; i < total; i += blockDim.x) out[i] = 0.0f;
        for (int i = tid; i < rows * (stride - d.l2); i += blockDim.x) out[(i / (stride - d.l2)) * stride + d.l2 + i % (stride - d.l2)] = 0.0f;
    }
    const int c = tid & 31, jj = slab * 32 + c;
    if (jj >= d.l2) return;
    for (int k = tid >> 5; k < rows; k += 8) {
        const int kk = min(k, m);                                   // intervals beyond the last finite breakpoint repeat it (never selected)
        float a;
        if (m == 0) a = 0.0f;
        else if (kk == 0) a = sorted[0] - fmaxf(1.0f, fabsf(sorted[0]));
        else if (kk == m) a = sorted[m - 1] + fmaxf(1.0f, fabsf(sorted[m - 1]));
        else a = 0.5f * (sorted[kk - 1] + sorted[kk]);
        float acc = 0.0f;
        for (int f = 0; f < la; ++f)
            if (fmaf(a, wa[f], ba[f]) > 0.0f) acc += col[f][c];
        out[k * stride + jj] = acc;
    }
}

// Everything a learn step prepares before its first network pass, in ONE launch (three dependent small launches cost ~40 us of
// launch gaps at C2): the V table of the critic-action pass (first blocks: the longest dependent chain), the BN-folded 16-bit
// weight packs of the four networks, and the hi/lo-split x_ext operand of the dgrad kernels.
struct PrepArgs {
    FoldJobs jobs;
    int A, l2, f16;
    unsigned fold_gx, fold_gy, n_fold, n_vtab, vtab_gy, fold_z0;
    const float* critic; int64_t cstride; CriticOff co; avd_net_dims d; float* vtab; int v_rows, v_stride, v_total;
    const float* s; int64_t s_rs; const float* a; int64_t N; bf16* xextT; int64_t R, Rp;
};

__global__ void __launch_bounds__(256) learn_prep_kernel(const __grid_constant__ PrepArgs p) {
    const unsigned b = blockIdx.x;
    if (b < p.n_vtab) {
        critic_vtab_body(p.critic, p.cstride, p.co, p.d, p.vtab, p.v_rows, p.v_stride, p.v_total, (int)(b / p.vtab_gy), (int)(b % p.vtab_gy));
    } else if (b < p.n_vtab + p.n_fold) {
        const unsigned f = b - p.n_vtab;
        pack_fold4_body(p.jobs, p.A, p.l2, p.f16, (int)(f % p.fold_gx), (int)((f / p.fold_gx) % p.fold_gy), (int)(f / (p.fold_gx * p.fold_gy) + p.fold_z0));
    } else {
        xext_body(p.s, p.s_rs, p.a, p.d.ns, p.N, p.xextT, p.R, p.Rp, p.f16, (int64_t)(b - p.n_vtab - p.n_fold));
    }
}

// Actor backward tile of the learn step without a second forward pass: MODE_ACTOR_SAVE kept the sign bits of z2 + b2' and
// d(action)/d(pre-activation), the critic-action pass delivered d(-mean q)/d(action) per row, so
//   dq_n = dpi_n * dact_n,     dm[n][j] = dm_scale * dq_n [z2 + b2' > 0][n][j]      (trainer.py:503-506 through model.py:30-37)
// is elementwise: 24 B read and 256 B written per row (HBM-bound) instead of the 118 us tensor-core pass it replaces.
// 16 threads per row (8 columns = one 16-byte store each); grid (row blocks, agents); sum_n dq_n accumulated per agent.
template <bool F16>
__global__ void __launch_bounds__(256) actor_dm_kernel(const float* __restrict__ dpi, const float* __restrict__ dact, const uint32_t* __restrict__ mask2,
                                                       bf16* __restrict__ DZ, float* __restrict__ sdq, int64_t R, float dm_scale) {
    pdl_wait();
    pdl_launch_dependents();
    const int agent = blockIdx.y;
    const int seg = threadIdx.x & 15;
    float acc = 0.0f;
    // Four rows per thread and iteration, all twelve loads issued before the first store.  Stand-alone (8 CTAs per SM) this is slower than
    // one row per iteration; beside a persistent tensor-core CTA, where only one or two of these CTAs fit on an SM, the loads in
    // flight per thread are what keeps the HBM write stream going.
    constexpr int UNR = 4;
    const int64_t stride = (int64_t)gridDim.x * 16;
    for (int64_t r0 = (int64_t)blockIdx.x * 16 + (threadIdx.x >> 4); r0 < R; r0 += stride * UNR) {
        float dq[UNR];
        uint32_t bits[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int64_t r = r0 + u * stride;
            const int64_t n = (int64_t)agent * R + (r < R ? r : R - 1);
            dq[u] = __ldg(dpi + n) * __ldg(dact + n);
            bits[u] = __ldg(mask2 + n * 4 + (seg >> 2)) << ((seg & 3) * 8);      // column 8 seg + k at bit 31 - k
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int64_t r = r0 + u * stride;
            if (r < R) {
                if (seg == 0) acc += dq[u];
                const float dqs = dq[u] * dm_scale;
                uint32_t pk[4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    pk[k] = umma::pack_x2<F16>((bits[u] & (0x80000000u >> (2 * k))) ? 0.0f : dqs, (bits[u] & (0x80000000u >> (2 * k + 1))) ? 0.0f : dqs);
                *reinterpret_cast<uint4*>(DZ + ((int64_t)agent * R + r) * 128 + seg * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
        }
    }
    __shared__ float red[8];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k];
        atomicAdd(sdq + agent, t);
    }
}

// Unfold the gradients of the BN-folded formulation into the Keras trainable tensors (one warp per layer-1 feature f).
// In:  G2[f][j] = sum_n r1[n][f] dz2[n][j] and G1[f][16] as `ncta` partial slices per agent (one per persistent CTA of the
//      wgrad / dgrad kernels, summed here),  G[ob2 + j] = db2[j]  (dgrad kernel).
// Out: dW2[f][j] = sc1[f] G2[f][j] + sh1[f] db2[j];   dsh1[f] = sum_j W2[f][j] db2[j];   dsc1[f] = sum_j W2[f][j] G2[f][j];
//      dbeta1 = dsh1;   dgamma1 = inv1 (dsc1 - mu1 dsh1);   dW1 / db1 from G1.          (trainer.py:498, 506; model.py:19-33, 62-77)
struct UnfoldOff {
    FoldOff f;
    int64_t W1[2], b1[2];     // layer-1 kernel / bias of the state columns [0] ([ns][l1]) and of the action columns [1] ([la])
};

struct HeadOff { int64_t g2, be2, mu2, var2, W3, b3; };

constexpr int kUnfoldWarps = 4;      // 128-thread CTAs: 16 per SM, so that the F x A <= 320 x 4 CTAs of the C2 case are a single wave

__global__ void __launch_bounds__(32 * kUnfoldWarps) unfold_kernel(const float* __restrict__ params, int64_t pstride, float* __restrict__ grads, int64_t gstride,
                                                     const float* __restrict__ G2, int64_t g2_agent_stride, int64_t g2_cta_stride,
                                                     const float* __restrict__ G1, int ncta, UnfoldOff o, int F, int Fp, int l2, int ns,
                                                     const float* __restrict__ dbm, const float* __restrict__ b2f, float* __restrict__ U, HeadOff ho,
                                                     const float* __restrict__ sdq, int* __restrict__ ticket, const float* __restrict__ wscale, int f16,
                                                     float inv_dm) {
    pdl_wait();                  // partial slices of the wgrad / dgrad launches
    pdl_launch_dependents();
    // one CTA per (feature f, agent); its warps split the partial slices between them (slice w, w + kUnfoldWarps, ...) so that
    // every load is independent and 64 warps per SM hide the L2 / HBM latency, then combine through shared memory
    const int agent = blockIdx.y;
    const int f = blockIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __shared__ float red[kUnfoldWarps][128 + 16];
    const float* g2row = G2 + (int64_t)agent * g2_agent_stride + (int64_t)f * l2;
    const float* g1row = G1 + ((int64_t)agent * ncta * Fp + f) * 16;
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, acc1 = 0.0f;
#pragma unroll 5
    for (int sl = wid; sl < ncta; sl += kUnfoldWarps) {
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            const int j = lane + 32 * jj;
            if (j < l2) acc[jj] += __ldg(g2row + (int64_t)sl * g2_cta_stride + j);
        }
        if (lane < 16) acc1 += __ldg(g1row + (int64_t)sl * Fp * 16 + lane);
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) red[wid][lane + 32 * jj] = acc[jj];
    if (lane < 16) red[wid][128 + lane] = acc1;
    __syncthreads();
    if (wid != 0) return;
    const float* P = params + (int64_t)agent * pstride;
    float* G = grads + (int64_t)agent * gstride;
    const bool st = f < o.f.l1;
    const int c = st ? f : f - o.f.l1;
    const int64_t og = st ? o.f.g[0] : o.f.g[1], obe = st ? o.f.be[0] : o.f.be[1], ob1 = st ? o.b1[0] : o.b1[1];
    const float inv = 1.0f / sqrtf(P[(st ? o.f.var[0] : o.f.var[1]) + c] + kBnEps);
    const float sc = P[og + c] * inv;
    const float mu = P[(st ? o.f.mu[0] : o.f.mu[1]) + c];
    const float sh = P[obe + c] - mu * sc;
    // The backward tile is dm = dq [z2 + b2' > 0] (avd_fused3.cu), so the sums arrive without the head weight:
    //   G2m = r1^T dm,  dbm = sum_n dm   =>   G2 = G2m diag(w3'),  db2 = w3' dbm,   w3' = sc2 w3
    // and the head-weight sum  U[j] = sum_n dq_n relu(z2 + b2')[n][j] = sum_f W2'[f][j] G2m[f][j] + b2'[j] dbm[j]  falls out of the
    // same data (z2 = r1 W2'^T with the bf16-rounded W2' of the forward pass): every CTA adds its feature's term.
    float dsc = 0.0f, dsh = 0.0f;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
        const int j = lane + 32 * jj;
        if (j < l2) {
            float g2m = 0.0f;
#pragma unroll
            for (int w = 0; w < kUnfoldWarps; ++w) g2m += red[w][j];
            g2m *= inv_dm;           // the fp16 backward tile carried the power-of-two factor dm_scale (avd_fused3.cu); 1 for bf16
            const float w3p = P[ho.W3 + j] * P[ho.g2 + j] / sqrtf(P[ho.var2 + j] + kBnEps);
            const float dbmj = dbm[(int64_t)agent * l2 + j] * inv_dm;
            const float g2 = w3p * g2m, db2 = w3p * dbmj;
            const int64_t i = o.f.W2 + (int64_t)f * l2 + j;
            const float w2 = P[i];
            dsc = fmaf(w2, g2, dsc);
            dsh = fmaf(w2, db2, dsh);
            G[i] = fmaf(sc, g2, sh * db2);
            float uj = round_op16(sc * w2, f16) * g2m;
            if (f == 0) {
                uj = fmaf(b2f[(int64_t)agent * l2 + j], dbmj, uj);
                G[o.f.b2 + j] = db2;
            }
            atomicAdd(U + (int64_t)agent * l2 + j, uj);
        }
    }
    dsc = warp_sum(dsc);
    dsh = warp_sum(dsh);
    float g1k = 0.0f;
    if (lane < 16) {
#pragma unroll
        for (int w = 0; w < kUnfoldWarps; ++w) g1k += red[w][128 + lane];
        g1k *= wscale ? wscale[agent] * inv_dm : inv_dm;       // the fp16 dgrad operands carried the power-of-two scales s (W2'') and dm_scale
    }
    float g1[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) g1[k] = __shfl_sync(0xffffffffu, g1k, k);
    if (lane == 0) {
        G[obe + c] = dsh;
        G[og + c] = inv * (dsc - mu * dsh);
        G[ob1 + c] = g1[5];
        if (st) {
            for (int x = 0; x < ns && x < 4; ++x) G[o.W1[0] + (int64_t)x * o.f.l1 + c] = g1[x] + g1[8 + x];
        } else {
            G[o.W1[1] + c] = g1[4] + g1[12];
        }
    }
    // ---- head / BatchNorm-2 gradients: they need the COMPLETE U of the agent, so the CTA that takes the last of the agent's F
    // tickets does them (every CTA's atomics on U precede its ticket; the counters are zeroed with the other accumulators)
    __threadfence();
    int last = 0;
    if (lane == 0) last = atomicAdd(ticket + agent, 1) == F - 1;
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    __threadfence();
    const float sd = __ldcg(sdq + agent);
    for (int j = lane; j < l2; j += 32) {
        const float inv2 = 1.0f / sqrtf(P[ho.var2 + j] + kBnEps);
        const float sc2 = P[ho.g2 + j] * inv2, mu2 = P[ho.mu2 + j];
        const float sh2 = P[ho.be2 + j] - mu2 * sc2;
        const float w3 = P[ho.W3 + j], u = __ldcg(U + (int64_t)agent * l2 + j);
        G[ho.W3 + j] = fmaf(sc2, u, sh2 * sd);           // dW3 = sc2 U + sh2 sum dq
        G[ho.g2 + j] = w3 * inv2 * (u - mu2 * sd);
        G[ho.be2 + j] = w3 * sd;
    }
    if (lane == 0) G[ho.b3] = sd;
}

// Head / BN2 gradients from the sums the fused backward pass accumulates (avd_fused3.cu):
//   U[j] = sum_n dq_n relu(z2)[n][j],  sd = sum_n dq_n,   h2 = relu(z2) sc2 + sh2,   q = h2 . w3 + b3
//   dW3 = sc2 U + sh2 sd;   dgamma2 = w3 inv2 (U - mu2 sd);   dbeta2 = w3 sd;   db3 = sd     (db2 comes out of the wgrad GEMM)

// ------------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------------
struct Workspace {
    float *H, *H1a, *Z, *Za, *DZ, *DH, *a2, *y, *q, *dpi;
    bf16 *cW2b, *cW2T, *tcW2T, *aW2b, *aW2T, *taW2T;   // packed weights (precision 1: bf16; precision 2: fp16; precision 3: three bf16 planes)
    float* vtab;               // [A][fused3::vtab_floats()] V table + breakpoints of the critic-action pass
    float* wscale;             // precision 2: [2][A] 1 / s of the critic [0] and actor [1] W2'' / T packs
    uint32_t* mask2;           // [N][4] sign bits of the actor's z2 + b2' (MODE_ACTOR_SAVE -> actor_dm_kernel)
    float* dact;               // [N] d(action)/d(pre-activation) of the actor
    // BN-folded tensor-core path: sign masks of z1, [x_hi | 1 | x_lo] operand, layer-1 weight-gradient accumulator, folded biases
    uint32_t* mask;
    // The actor's backward chain (tile, layer-1 sign masks, partial slices) has buffers of its own, so that it can overlap the critic's
    // chain on the side stream: DZa is the second half of the DZ region (sized for fp32 tiles, the fused path writes 16-bit ones).
    bf16* DZa;
    uint32_t* mask_a;          // [N][8]
    float *G1a, *G2part_a;
    bf16* xextT;               // [A][16][Rp], Rp = R rounded up to 64
    float *G1, *G2part, *c_b2f, *tc_b2f, *a_b2f, *ta_b2f;     // G1 / G2part: one partial slice per persistent CTA (<= max(A, #SMs) slices)
    float *U, *sdq;            // [2][A][l2], [2][A]: head-gradient sums of the critic [0] and actor [1] backward passes
    float* dbm;                // [2][A][l2]: sum_n dm[n][j] of the two backward passes (db2 = w3' dbm)
    int* ticket;               // [2][A]: CTAs of the unfold kernel that have finished (the last one unfolds the head)
    static constexpr int kMaskWords = 10, kFp = 320, kG2Rows = 384;
    // fused: the persistent tensor-core kernels keep every activation on chip -- only the dz2 tile (DZ) of the fp32 activation
    // buffers exists then (C2: 0.9 GB instead of 5.4 GB of workspace, C4: 3.5 GB instead of 21 GB)
    // planes = 3 (precision 3): the GEMM operands H, H1a, DZ and the six weight packs hold three bf16 planes, 6 B per element
    static int64_t bytes(const avd_net_dims& d, int64_t A, int64_t N, bool fused, int planes) {
        const int64_t F = d.l1 + d.la;
        int64_t acts = N * (fused ? (int64_t)d.l2 : 2 * F + d.l1 + 3 * (int64_t)d.l2) * (int64_t)sizeof(float);
        if (planes == 3) acts += N * (F + d.l1 + d.l2) * 2;
        const int64_t packed = planes * A * (3 * F + 3 * (int64_t)d.l1) * d.l2 * (int64_t)sizeof(bf16) + (2 * A + 4 + A * (int64_t)fused3::vtab_floats()) * (int64_t)sizeof(float);
        const int64_t vecs = (5 + 4) * ((N + 3) / 4 * 4) * (int64_t)sizeof(float);
        const int64_t slices = std::max<int64_t>(A, sm_count());
        const int64_t fold = N * ((kMaskWords + 8) * 4 + 16 * 2) + A * (8 * (int64_t)d.l2 + 16) * (int64_t)sizeof(float) + A * 16 * 64 * 2 +
                             2 * slices * (kFp * 16 + kG2Rows * (int64_t)d.l2) * (int64_t)sizeof(float);
        return acts + packed + vecs + fold + 1024;
    }
    void carve(void* base_, const avd_net_dims& d, int64_t A, int64_t N, bool fused, int planes) {
        const int64_t F = d.l1 + d.la;
        float* p = reinterpret_cast<float*>(((uintptr_t)base_ + 255) & ~(uintptr_t)255);
        // floats taken by a GEMM-operand buffer of n elements: fp32 / one 16-bit copy (planes = 1) or three bf16 planes
        auto opnd = [planes](int64_t n) { return planes == 3 ? n * 3 / 2 : n; };
        H = DH = H1a = Z = Za = nullptr;
        if (!fused) {
            H = p; p += opnd(N * F);
            DH = p; p += N * F;
            H1a = p; p += opnd(N * d.l1);
            Z = p; p += N * d.l2;
            Za = p; p += N * d.l2;
        }
        DZ = p; p += opnd(N * d.l2);
        DZa = reinterpret_cast<bf16*>(DZ) + N * d.l2;
        bf16* b = reinterpret_cast<bf16*>(p);
        cW2b = b; b += planes * A * F * d.l2;
        cW2T = b; b += planes * A * F * d.l2;
        tcW2T = b; b += planes * A * F * d.l2;
        aW2b = b; b += planes * A * (int64_t)d.l1 * d.l2;
        aW2T = b; b += planes * A * (int64_t)d.l1 * d.l2;
        taW2T = b; b += planes * A * (int64_t)d.l1 * d.l2;
        p = reinterpret_cast<float*>(((uintptr_t)b + 15) & ~(uintptr_t)15);
        wscale = p; p += (2 * A + 3) / 4 * 4;
        vtab = p; p += A * (int64_t)fused3::vtab_floats();
        const int64_t Np = (N + 3) / 4 * 4;
        a2 = p; p += Np;
        y = p; p += Np;
        q = p; p += Np;
        dpi = p; p += Np;
        dact = p; p += Np;
        mask2 = reinterpret_cast<uint32_t*>(p); p += 4 * Np;
        const int64_t slices = std::max<int64_t>(A, sm_count());
        G1 = p; p += slices * kFp * 16;
        G2part = p; p += slices * kG2Rows * d.l2;
        G1a = p; p += slices * kFp * 16;
        G2part_a = p; p += slices * kG2Rows * d.l2;
        c_b2f = p; p += A * d.l2;
        tc_b2f = p; p += A * d.l2;
        a_b2f = p; p += A * d.l2;
        ta_b2f = p; p += A * d.l2;
        dbm = p; p += 2 * A * d.l2;
        ticket = reinterpret_cast<int*>(p); p += (2 * A + 3) / 4 * 4;
        U = p; p += 2 * A * d.l2;
        sdq = p; p += (2 * A + 3) / 4 * 4;
        mask = reinterpret_cast<uint32_t*>(p); p += N * kMaskWords;
        mask_a = reinterpret_cast<uint32_t*>(p); p += N * 8;
        xextT = reinterpret_cast<bf16*>(((uintptr_t)p + 15) & ~(uintptr_t)15);
    }
};

static int check_dims(const avd_net_dims* d, int precision = 0) {
    AVD_REQUIRE(d, "null dims");
    AVD_REQUIRE(d->ns >= 1 && d->ns <= 8, "ns=%d outside 1..8", d->ns);
    AVD_REQUIRE(d->l1 >= 4 && d->la >= 4 && d->l1 % 4 == 0 && d->la % 4 == 0 && d->la <= 64,
                "layer sizes must be multiples of 4 and la <= 64 (l1=%d, la=%d)", d->l1, d->la);
    AVD_REQUIRE(precision >= 0 && precision <= 3, "precision must be 0 (fp32 SIMT), 1 (bf16 tcgen05), 2 (fp16 tcgen05) or 3 (split bf16 tcgen05)");
    if (d->l2 != 32 && d->l2 != 64 && d->l2 != 96 && d->l2 != 128) {
        set_error("layer2 size %d not supported (32, 64, 96 or 128)", d->l2);
        return AVD_ERR_UNSUPPORTED;
    }
    if (precision >= 1 && (d->l1 % 8 || d->la % 8 || d->l2 % 8)) {
        set_error("precision 1 / 2 / 3 need layer sizes that are multiples of 8 (TMA 16-byte pitch)");
        return AVD_ERR_UNSUPPORTED;
    }
    return AVD_OK;
}

template <int MODE, typename TDZ>
static void launch_head_t(const HeadArgs& h, int l2, dim3 grid, cudaStream_t st) {
    switch (l2 / 32) {
        case 1: head_kernel<MODE, 1, TDZ><<<grid, 256, 0, st>>>(h); break;
        case 2: head_kernel<MODE, 2, TDZ><<<grid, 256, 0, st>>>(h); break;
        case 3: head_kernel<MODE, 3, TDZ><<<grid, 256, 0, st>>>(h); break;
        default: head_kernel<MODE, 4, TDZ><<<grid, 256, 0, st>>>(h); break;
    }
}

// prec: the learn step's precision, which decides the operand format of the backward tile DZ
template <int MODE>
static int launch_head(const HeadArgs& h, int l2, int A, cudaStream_t st, int prec = 0) {
    dim3 grid((unsigned)((h.R + 63) / 64), A);
    HeadArgs hp = h;
    hp.dz_plane = (int64_t)A * h.R * l2;
    with_operand(prec, h.DZ, hp.dz_plane, [&](auto dz) { launch_head_t<MODE, decltype(dz)>(hp, l2, grid, st); });
    AVD_LAUNCH_OK();
    return AVD_OK;
}

static HeadArgs actor_head(const avd_net_dims& d, const float* params, const float* Z, int64_t R, float high) {
    const ActorOff o = actor_off(d);
    HeadArgs h = {};
    h.params = params; h.pstride = o.total;
    h.o_b2 = o.b2; h.o_g2 = o.g2; h.o_be2 = o.be2; h.o_mu2 = o.mu2; h.o_var2 = o.var2; h.o_W3 = o.W3; h.o_b3 = o.b3;
    h.Z = Z; h.R = R; h.high = high;
    return h;
}

static HeadArgs critic_head(const avd_net_dims& d, const float* params, const float* Z, int64_t R) {
    const CriticOff o = critic_off(d);
    HeadArgs h = {};
    h.params = params; h.pstride = o.total;
    h.o_b2 = o.b2; h.o_g2 = o.g2; h.o_be2 = o.be2; h.o_mu2 = o.mu2; h.o_var2 = o.var2; h.o_W3 = o.W3; h.o_b3 = o.b3;
    h.Z = Z; h.R = R;
    return h;
}

// Everything a pass needs; `prec` selects fp32 SIMT tiles or bf16 tcgen05 for the three big contractions.
struct Pass {
    avd_net_dims d;
    int A, prec;
    int64_t R;
    cudaStream_t st;

    bool f16() const { return prec == 2; }     // fp16 layer-2 operands in the fused tensor-core kernels

    // the fields every fused pass sets; the caller adds those of its mode
    fused3::RunArgs fused_args(fused3::Mode mode, const float* params, const bf16* W2T, const float* b2f, const float* s, int64_t s_rs) const {
        const bool actor = mode == fused3::MODE_ACTOR_OUT || mode == fused3::MODE_ACTOR_SAVE;
        fused3::RunArgs a;
        a.mode = mode; a.f16 = f16(); a.d = d; a.A = A; a.R = R;
        a.params = params; a.pstride = actor ? actor_off(d).total : critic_off(d).total;
        a.W2T = W2T; a.b2f = b2f; a.s = s; a.s_rs = s_rs;
        return a;
    }

    dim3 l1_grid() const { return dim3((unsigned)((R + kL1Rows - 1) / kL1Rows), A); }

    // layer 1 (+BN) of the actor (critic=false) or critic (true) into H ([N][F] in the operand format)
    int layer1(bool critic, const float* params, const float* s, int64_t s_rs, int64_t s_cs, const float* act, void* H) const {
        const int64_t ps = critic ? critic_off(d).total : actor_off(d).total;
        with_operand(prec, H, (int64_t)A * R * (critic ? d.l1 + d.la : d.l1), [&](auto o) {
            if (critic) l1_forward_kernel<true, decltype(o)><<<l1_grid(), 128, 0, st>>>(d, params, ps, s, s_rs, s_cs, act, R, o);
            else l1_forward_kernel<false, decltype(o)><<<l1_grid(), 128, 0, st>>>(d, params, ps, s, s_rs, s_cs, act, R, o);
        });
        AVD_LAUNCH_OK();
        return AVD_OK;
    }

    // 16-bit layer-2 kernels W2b / W2T of A agents in the operand format of precision 1, 2 or 3 (planes of A*F*l2 elements)
    int pack(const float* params, int64_t pstride, int64_t oW2, int F, bf16* W2b, bf16* W2T) const {
        const dim3 grid((unsigned)((F * d.l2 + 255) / 256), A);
        const int64_t plane = (int64_t)A * F * d.l2;
        with_operand(prec, W2T, plane, [&](auto o) {
            using T = decltype(o);
            if constexpr (!std::is_same<T, float*>::value)
                pack_w2_kernel<T><<<grid, 256, 0, st>>>(params, pstride, oW2, F, d.l2, as_operand<T>(W2b, plane), o);
        });
        AVD_LAUNCH_OK();
        return AVD_OK;
    }

    // BN-folded packing (fused tensor-core path)
    int pack_fold(bool critic, const float* params, bf16* W2b, bf16* W2T, float* b2f) const {
        const FoldOff o = fold_off(critic);
        const int F = critic ? d.l1 + d.la : d.l1;
        const int64_t ps = critic ? critic_off(d).total : actor_off(d).total;
        pack_fold_kernel<<<dim3((unsigned)((d.l2 + 31) / 32), (unsigned)((F + 7) / 8), A), 256, 0, st>>>(params, ps, o, F, d.l2, W2b, W2T, b2f, f16() ? 1 : 0);
        AVD_LAUNCH_OK();
        return AVD_OK;
    }

    // all four networks of a learn step in one launch
    // wscale[i] (fp16 only, nullable): [A] 1 / s of job i's W2b pack.
    int pack_fold4(FoldJobs& jobs, int& Fmax, int njobs, const float* const params[], const bool critic[], bf16* const W2b[], bf16* const W2T[],
                   float* const b2f[], float* const wscale[]) const {
        jobs = FoldJobs{};
        Fmax = 0;
        for (int i = 0; i < njobs; ++i) {
            FoldJob& jb = jobs.j[i];
            jb.params = params[i];
            jb.pstride = critic[i] ? critic_off(d).total : actor_off(d).total;
            jb.o = fold_off(critic[i]);
            if (critic[i]) { const CriticOff c = critic_off(d); jb.g2 = c.g2; jb.var2 = c.var2; jb.W3 = c.W3; }
            else { const ActorOff a = actor_off(d); jb.g2 = a.g2; jb.var2 = a.var2; jb.W3 = a.W3; }
            jb.F = critic[i] ? d.l1 + d.la : d.l1;
            jb.W2b = W2b[i]; jb.W2T = W2T[i]; jb.b2f = b2f[i]; jb.wscale = wscale[i];
            Fmax = std::max(Fmax, jb.F);
        }
        return AVD_OK;
    }

    FoldOff fold_off(bool critic) const {
        FoldOff o;
        if (critic) {
            const CriticOff c = critic_off(d);
            o.W2 = c.W2; o.b2 = c.b2; o.l1 = d.l1;
            o.g[0] = c.gs; o.be[0] = c.bes; o.mu[0] = c.mus; o.var[0] = c.vars;
            o.g[1] = c.ga; o.be[1] = c.bea; o.mu[1] = c.mua; o.var[1] = c.vara;
        } else {
            const ActorOff a = actor_off(d);
            o.W2 = a.W2; o.b2 = a.b2; o.l1 = d.l1;
            for (int k = 0; k < 2; ++k) { o.g[k] = a.g1; o.be[k] = a.be1; o.mu[k] = a.mu1; o.var[k] = a.var1; }
        }
        return o;
    }

    // fused dgrad + layer-1 weight gradient (avd_dgrad3.cu), then unfold.  G2part holds the partial G2 slices the wgrad kernel
    // (avd_wgrad3.cu) stored before: [A][ncta][384][l2].
    int dgrad3_only(const bf16* DZ, const bf16* W2b, int F, int Fp, const uint32_t* mask, int mask_words, const bf16* xextT, float* G1, float* dbm) const {
        return dgrad3::run(f16(), A, R, F, DZ, W2b, mask, mask_words, xextT, (R + 63) / 64 * 64, G1, Fp, dbm, d.l2, st);
    }
    int unfold(bool critic, const float* params, int F, int Fp, float* G1, const float* G2part, float* grads, float* dbm, const float* b2f, float* U,
               const float* sdq, int* ticket, const float* wscale, float dm_scale) const {
        const int64_t gs = critic ? critic_off(d).n_train : actor_off(d).n_train;
        const int ncta = ctas_per_agent(A, R);
        UnfoldOff u;
        u.f = fold_off(critic);
        int64_t ps;
        HeadOff ho;
        if (critic) {
            const CriticOff c = critic_off(d);
            u.W1[0] = c.Ws; u.b1[0] = c.bs; u.W1[1] = c.Wa; u.b1[1] = c.ba; ps = c.total;
            ho = HeadOff{c.g2, c.be2, c.mu2, c.var2, c.W3, c.b3};
        } else {
            const ActorOff a = actor_off(d);
            u.W1[0] = u.W1[1] = a.W1; u.b1[0] = u.b1[1] = a.b1; ps = a.total;
            ho = HeadOff{a.g2, a.be2, a.mu2, a.var2, a.W3, a.b3};
        }
        AVD_CUDA_OK(launch_pdl(unfold_kernel, dim3((unsigned)F, (unsigned)A), dim3(32 * kUnfoldWarps), 0, st, params, ps, grads, gs, G2part,
                               (int64_t)ncta * Workspace::kG2Rows * d.l2, (int64_t)Workspace::kG2Rows * d.l2, G1, ncta, u, F, Fp, d.l2, d.ns, (const float*)dbm, b2f, U, ho, sdq, ticket,
                               f16() ? wscale : (const float*)nullptr, f16() ? 1 : 0, 1.0f / dm_scale));
        AVD_LAUNCH_OK();
        return AVD_OK;
    }

    // Z[a] (R x l2) = H[a] (R x F) . W2[a] (F x l2)
    int forward(const void* H, int F, const float* params, int64_t pstride, int64_t oW2, const bf16* W2T, float* Z) const {
        if (operand_format(prec) != OPND_F32)
            return umma::gemm_bf16(operand_planes(prec), 0, A, (int)R, d.l2, F, H, F, R * F, W2T, F, (int64_t)d.l2 * F, Z, d.l2, R * d.l2, 1, st);
        GemmArgs g = {};
        g.A = (const float*)H; g.a_m = F; g.a_k = 1; g.a_batch = R * F;
        g.B = params + oW2; g.b_k = d.l2; g.b_n = 1; g.b_batch = pstride;
        g.C = Z; g.c_m = d.l2; g.c_n = 1; g.c_batch = R * d.l2;
        g.M = (int)R; g.N = d.l2; g.K = F; g.splitk = 1;
        return launch_sgemm(g, A, st);
    }

    // dW2[a] (F x l2) += H[a]^T . DZ[a]   (contraction over the R rows, split over CTAs, atomics into zeroed grads)
    int wgrad(const void* H, int F, const void* DZ, float* grads, int64_t gstride, int64_t oW2) const {
        const int tiles = ((F + (prec ? 127 : 63)) / (prec ? 128 : 64)) * ((d.l2 + (prec ? 127 : 63)) / (prec ? 128 : 64)) * A;
        const int64_t chunk = prec ? 64 : 256;
        int split = (int)std::min<int64_t>((R + chunk - 1) / chunk, std::max(1, 4 * sm_count() / std::max(1, tiles)));
        split = std::max(1, split);
        if (operand_format(prec) != OPND_F32)
            return umma::gemm_bf16(operand_planes(prec), 1, A, F, d.l2, (int)R, H, F, R * F, DZ, d.l2, R * d.l2, grads + oW2, d.l2, gstride, split, st);
        GemmArgs g = {};
        g.A = (const float*)H; g.a_m = 1; g.a_k = F; g.a_batch = R * F;
        g.B = (const float*)DZ; g.b_k = d.l2; g.b_n = 1; g.b_batch = R * d.l2;
        g.C = grads + oW2; g.c_m = d.l2; g.c_n = 1; g.c_batch = gstride;
        g.M = F; g.N = d.l2; g.K = (int)R; g.splitk = split;
        return launch_sgemm(g, A, st);
    }

    // DH[a] (R x Fsub) = DZ[a] (R x l2) . W2[a][f0:f0+Fsub, :]^T
    int dgrad(const void* DZ, const float* params, int64_t pstride, int64_t oW2, const bf16* W2b, int F, int f0, int Fsub, float* DH) const {
        if (operand_format(prec) != OPND_F32)
            return umma::gemm_bf16(operand_planes(prec), 0, A, (int)R, Fsub, d.l2, DZ, d.l2, R * d.l2, W2b + (int64_t)f0 * d.l2, d.l2,
                                   (int64_t)F * d.l2, DH, Fsub, R * Fsub, 1, st);
        GemmArgs g = {};
        g.A = (const float*)DZ; g.a_m = d.l2; g.a_k = 1; g.a_batch = R * d.l2;
        g.B = params + oW2 + (int64_t)f0 * d.l2; g.b_k = 1; g.b_n = d.l2; g.b_batch = pstride;
        g.C = DH; g.c_m = Fsub; g.c_n = 1; g.c_batch = R * Fsub;
        g.M = (int)R; g.N = Fsub; g.K = d.l2; g.splitk = 1;
        return launch_sgemm(g, A, st);
    }
};

}  // namespace avd

using namespace avd;

extern "C" int avd_ddpg_param_counts(const avd_net_dims* dims, int64_t* out4) {
    if (int rc = check_dims(dims)) return rc;
    AVD_REQUIRE(out4, "null out");
    const ActorOff a = actor_off(*dims);
    const CriticOff c = critic_off(*dims);
    out4[0] = a.n_train; out4[1] = a.total; out4[2] = c.n_train; out4[3] = c.total;
    return AVD_OK;
}

// the persistent fused kernels (avd_fused3.cu and friends) serve precision 1 and 2 at the dims they support
static bool fused_path(const avd_net_dims& d, int precision) { return (precision == 1 || precision == 2) && fused3::supported(d); }

extern "C" int64_t avd_ddpg_workspace_bytes(const avd_net_dims* dims, int32_t A, int64_t rows_per_agent, int32_t precision) {
    if (!dims || A < 0 || rows_per_agent < 0) return -1;
    return Workspace::bytes(*dims, A, (int64_t)A * rows_per_agent, fused_path(*dims, precision), operand_planes(precision));
}

// Workspace of the forward entry points, [H | Z | W2T]: layer-1 output in the operand format, layer-2 output (fp32), packed layer-2
// kernel (16-bit, one copy or three planes), from `base` rounded up to 256 bytes.
struct ForwardWorkspace {
    float *H, *Z;
    bf16* W2T;
    int64_t bytes;
};
static ForwardWorkspace forward_workspace(const avd_net_dims& d, int64_t A, int64_t R, bool critic, int precision, void* base) {
    const int64_t N = A * R, F = critic ? d.l1 + d.la : d.l1;
    const int64_t h = operand_bytes(precision, N * F), z = N * d.l2 * (int64_t)sizeof(float);
    const uintptr_t p = ((uintptr_t)base + 255) & ~(uintptr_t)255;
    ForwardWorkspace w;
    w.H = reinterpret_cast<float*>(p);
    w.Z = reinterpret_cast<float*>(p + h);
    w.W2T = reinterpret_cast<bf16*>(p + h + z);
    w.bytes = h + z + operand_planes(precision) * A * F * d.l2 * (int64_t)sizeof(bf16) + 512;
    return w;
}

extern "C" int64_t avd_forward_workspace_bytes(const avd_net_dims* dims, int32_t A, int64_t rows_per_agent, int32_t critic, int32_t precision) {
    if (!dims || A < 0 || rows_per_agent < 0) return -1;
    return forward_workspace(*dims, A, rows_per_agent, critic != 0, precision, nullptr).bytes;
}

#define AVD_TRY(expr)             \
    do {                          \
        int _rc = (expr);         \
        if (_rc) return _rc;      \
    } while (0)

extern "C" int avd_actor_forward(const avd_net_dims* dims, int32_t A, int64_t R, const float* actor_params, const float* s,
                                 int64_t s_rs, int64_t s_cs, float action_high, float* out, void* workspace,
                                 int64_t workspace_bytes, int32_t precision, void* stream) {
    AVD_TRY(check_dims(dims, precision));
    AVD_REQUIRE(actor_params && s && out && workspace, "null buffer");
    AVD_REQUIRE(A >= 0 && R >= 0, "bad sizes");
    const avd_net_dims d = *dims;
    const ForwardWorkspace w = forward_workspace(d, A, R, false, precision, workspace);
    AVD_REQUIRE(workspace_bytes >= w.bytes, "workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)w.bytes);
    if ((int64_t)A * R == 0) return AVD_OK;
    const Pass p{d, A, precision, R, (cudaStream_t)stream};
    const ActorOff o = actor_off(d);
    if (fused_path(d, precision)) {   // fused kernel: H / Z are never materialised, their space holds the folded bias
        AVD_TRY(p.pack_fold(false, actor_params, nullptr, w.W2T, w.H));
        fused3::RunArgs f = p.fused_args(fused3::MODE_ACTOR_OUT, actor_params, w.W2T, w.H, s, s_rs);
        f.s_cs = s_cs; f.high = action_high; f.out = out;
        return fused3::run(f, p.st);
    }
    if (precision) AVD_TRY(p.pack(actor_params, o.total, o.W2, d.l1, nullptr, w.W2T));
    AVD_TRY(p.layer1(false, actor_params, s, s_rs, s_cs, nullptr, w.H));
    AVD_TRY(p.forward(w.H, d.l1, actor_params, o.total, o.W2, w.W2T, w.Z));
    HeadArgs h = actor_head(d, actor_params, w.Z, R, action_high);
    h.out = out;
    return launch_head<HEAD_ACTOR_FWD>(h, d.l2, A, p.st);
}

extern "C" int avd_critic_forward(const avd_net_dims* dims, int32_t A, int64_t R, const float* critic_params, const float* s,
                                  const float* a, float* q, void* workspace, int64_t workspace_bytes, int32_t precision,
                                  void* stream) {
    AVD_TRY(check_dims(dims, precision));
    AVD_REQUIRE(critic_params && s && a && q && workspace, "null buffer");
    AVD_REQUIRE(A >= 0 && R >= 0, "bad sizes");
    const avd_net_dims d = *dims;
    const int F = d.l1 + d.la;
    const ForwardWorkspace w = forward_workspace(d, A, R, true, precision, workspace);
    AVD_REQUIRE(workspace_bytes >= w.bytes, "workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)w.bytes);
    if ((int64_t)A * R == 0) return AVD_OK;
    const Pass p{d, A, precision, R, (cudaStream_t)stream};
    const CriticOff o = critic_off(d);
    if (fused_path(d, precision)) {
        AVD_TRY(p.pack_fold(true, critic_params, nullptr, w.W2T, w.H));
        fused3::RunArgs f = p.fused_args(fused3::MODE_Q, critic_params, w.W2T, w.H, s, d.ns);
        f.act = a; f.out = q;
        return fused3::run(f, p.st);
    }
    if (precision) AVD_TRY(p.pack(critic_params, o.total, o.W2, F, nullptr, w.W2T));
    AVD_TRY(p.layer1(true, critic_params, s, d.ns, 1, a, w.H));
    AVD_TRY(p.forward(w.H, F, critic_params, o.total, o.W2, w.W2T, w.Z));
    HeadArgs h = critic_head(d, critic_params, w.Z, R);
    h.out = q;
    return launch_head<HEAD_CRITIC_Q>(h, d.l2, A, p.st);
}

extern "C" int avd_adam_apply(float* params, int64_t param_stride, const float* grads, int64_t grad_agent_stride, float* m, float* v,
                              int32_t* step, const uint8_t* apply_mask, int32_t A, int64_t n, float lr, float beta1, float beta2,
                              float eps, void* stream) {
    AVD_REQUIRE(params && grads && m && v && step, "null buffer");
    AVD_REQUIRE(A >= 0 && n >= 0 && param_stride >= n, "bad sizes");
    if (A == 0 || n == 0) return AVD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int gx = (int)std::min<int64_t>((n + 255) / 256, 64);
    adam_kernel<<<dim3(gx, A), 256, 0, st>>>(params, param_stride, grads, grad_agent_stride, m, v, step, apply_mask, n, lr, beta1, beta2, eps);
    AVD_LAUNCH_OK();
    step_increment_kernel<<<(A + 127) / 128, 128, 0, st>>>(step, apply_mask, A);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_adam_polyak_apply2(float* actor, float* t_actor, int64_t actor_total, const float* actor_grad, int64_t actor_gstride,
                                      float* actor_m, float* actor_v, int32_t* actor_step, int64_t actor_train, float actor_lr, float* critic,
                                      float* t_critic, int64_t critic_total, const float* critic_grad, int64_t critic_gstride, float* critic_m,
                                      float* critic_v, int32_t* critic_step, int64_t critic_train, float critic_lr, const uint8_t* apply_mask,
                                      int32_t A, float beta1, float beta2, float eps, float tau, const float* agent_hp, void* stream) {
    AVD_REQUIRE(actor && t_actor && actor_grad && actor_m && actor_v && actor_step && critic && t_critic && critic_grad && critic_m && critic_v &&
                    critic_step,
                "null buffer");
    AVD_REQUIRE(A >= 0 && actor_train >= 0 && actor_total >= actor_train && critic_train >= 0 && critic_total >= critic_train, "bad sizes");
    if (A == 0) return AVD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    AdamNets nets;
    nets.n[0] = AdamNet{critic, t_critic, critic_grad, critic_m, critic_v, critic_step, critic_total, critic_gstride, critic_train, critic_total, critic_lr};
    nets.n[1] = AdamNet{actor, t_actor, actor_grad, actor_m, actor_v, actor_step, actor_total, actor_gstride, actor_train, actor_total, actor_lr};
    const int64_t blocks = std::min<int64_t>((std::max(critic_total, actor_total) + 255) / 256, 1024);
    const dim3 grid((unsigned)blocks, (unsigned)A, 2);
    if (agent_hp) AVD_CUDA_OK(launch_pdl(adam_polyak2_kernel<true>, grid, dim3(256), 0, st, nets, apply_mask, beta1, beta2, eps, tau, agent_hp));
    else AVD_CUDA_OK(launch_pdl(adam_polyak2_kernel<false>, grid, dim3(256), 0, st, nets, apply_mask, beta1, beta2, eps, tau, agent_hp));
    AVD_LAUNCH_OK();
    AVD_CUDA_OK(launch_pdl(step_increment2_kernel, dim3((unsigned)((A + 127) / 128)), dim3(128), 0, st, actor_step, critic_step, apply_mask, (int)A));
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_polyak_update(float* target, const float* online, const uint8_t* apply_mask, int32_t A, int64_t n, float tau,
                                 void* stream) {
    AVD_REQUIRE(target && online, "null buffer");
    AVD_REQUIRE(A >= 0 && n >= 0, "bad sizes");
    if (A == 0 || n == 0) return AVD_OK;
    const int gx = (int)std::min<int64_t>((n + 255) / 256, 64);
    polyak_kernel<<<dim3(gx, A), 256, 0, (cudaStream_t)stream>>>(target, online, apply_mask, n, tau);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_fed_reduce(float* out, int64_t out_pitch, const float* in, int64_t pitch, int32_t n_systems, int32_t n_members,
                              int64_t member_stride_s, int64_t member_stride_x, const float* weights, const float* scale, int64_t n,
                              void* stream) {
    AVD_REQUIRE(out && in, "null buffer");
    AVD_REQUIRE(n_systems >= 0 && n_members >= 1 && n >= 0, "bad sizes");
    if (n_systems == 0 || n == 0) return AVD_OK;
    const int gx = (int)std::min<int64_t>((n + 255) / 256, 128);
    fed_reduce_kernel<<<dim3(gx, n_systems), 256, 0, (cudaStream_t)stream>>>(out, out_pitch, in, pitch, n_members, member_stride_s,
                                                                              member_stride_x, weights, scale, n);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_fed_reduce2(float* out, int64_t out_pitch, const float* in_a, int64_t pitch_a, int64_t na, const float* in_c, int64_t pitch_c,
                               int64_t nc, int32_t n_systems, int32_t n_members, int64_t member_stride_s, int64_t member_stride_x,
                               const float* weights, void* stream) {
    AVD_REQUIRE(out && in_a && in_c, "null buffer");
    AVD_REQUIRE(n_systems >= 0 && n_members >= 1 && na >= 0 && nc >= 0 && out_pitch > na + nc, "bad sizes");
    if (n_systems == 0) return AVD_OK;
    const int gx = (int)std::min<int64_t>((na + nc + 256) / 256, 128);
    fed_reduce2_kernel<<<dim3(gx, n_systems), 256, 0, (cudaStream_t)stream>>>(out, out_pitch, in_a, pitch_a, na, in_c, pitch_c, nc, n_members,
                                                                               member_stride_s, member_stride_x, weights);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_fed_broadcast2(float* out_a, int64_t pitch_a, int64_t na, float* out_c, int64_t pitch_c, int64_t nc, const float* in,
                                  int64_t in_pitch, int32_t n_systems, int32_t n_members, int64_t member_stride_s, int64_t member_stride_x,
                                  const uint8_t* apply_mask, void* stream) {
    AVD_REQUIRE(out_a && out_c && in, "null buffer");
    AVD_REQUIRE(n_systems >= 0 && n_members >= 1 && na >= 0 && nc >= 0, "bad sizes");
    if (n_systems == 0 || na + nc == 0) return AVD_OK;
    const int gx = (int)std::min<int64_t>((na + nc + 255) / 256, 64);
    fed_broadcast2_kernel<<<dim3(gx, n_systems, n_members), 256, 0, (cudaStream_t)stream>>>(out_a, pitch_a, na, out_c, pitch_c, nc, in, in_pitch,
                                                                                             n_members, member_stride_s, member_stride_x, apply_mask);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_fed_weights_from_history(const float* ep_hist, int32_t window, int32_t M, int64_t G, int64_t E, float* out_w,
                                            int32_t transpose, void* stream) {
    AVD_REQUIRE(ep_hist && out_w, "null buffer");
    AVD_REQUIRE(window >= 1 && M >= 1 && G >= 1 && E >= 1 && (int64_t)M * G < (1 << 30), "bad sizes");
    fed_weights_kernel<<<(unsigned)(M * G), 256, 0, (cudaStream_t)stream>>>(ep_hist, window, M, G, E, out_w, transpose);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_fed_finalize(float* buf, int64_t pitch, int32_t n_systems, int64_t n, void* stream) {
    AVD_REQUIRE(buf && n_systems >= 0 && n >= 0 && pitch > n, "bad args");
    if (n_systems == 0 || n == 0) return AVD_OK;
    const int gx = (int)std::min<int64_t>((n + 255) / 256, 128);
    fed_finalize_kernel<<<dim3(gx, n_systems), 256, 0, (cudaStream_t)stream>>>(buf, pitch, n);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_fed_broadcast(float* out, int64_t out_pitch, const float* in, int64_t in_pitch, int32_t n_systems, int32_t n_members,
                                 int64_t member_stride_s, int64_t member_stride_x, const uint8_t* apply_mask, int64_t n, void* stream) {
    AVD_REQUIRE(out && in, "null buffer");
    AVD_REQUIRE(n_systems >= 0 && n_members >= 1 && n >= 0, "bad sizes");
    if (n_systems == 0 || n == 0) return AVD_OK;
    const int gx = (int)std::min<int64_t>((n + 255) / 256, 64);
    fed_broadcast_kernel<<<dim3(gx, n_systems, n_members), 256, 0, (cudaStream_t)stream>>>(out, out_pitch, in, in_pitch, n_members,
                                                                                            member_stride_s, member_stride_x, apply_mask, n);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

// Adam on both nets, then Polyak of the targets                                       trainer.py:345-356
static int apply_local_updates(const avd_learn_io* io, void* stream) {
    if (!io->apply_updates) return AVD_OK;
    const ActorOff ao = actor_off(io->dims);
    const CriticOff co = critic_off(io->dims);
    const int A = io->A;
    AVD_TRY(avd_adam_polyak_apply2(io->actor, io->t_actor, ao.total, io->actor_grad, ao.n_train, io->actor_m, io->actor_v, io->actor_t, ao.n_train,
                                   io->actor_lr, io->critic, io->t_critic, co.total, io->critic_grad, co.n_train, io->critic_m, io->critic_v,
                                   io->critic_t, co.n_train, io->critic_lr, io->apply_mask, A, io->adam_beta1, io->adam_beta2, io->adam_eps,
                                   io->tau, io->agent_hp, stream));
    return AVD_OK;
}

// The learn step on the third-generation kernels: six persistent pass launches (avd_fused3.cu) cover every forward pass,
// both head backwards and the critic -> actor link; per differentiated net only dz2 (256 B per row) and the ReLU sign masks
// (40 B) go to HBM, for the layer-2 weight gradient (avd_wgrad3.cu, recomputes r1 on chip) and the fused dgrad + layer-1
// weight gradient + layer-2 bias gradient (avd_dgrad3.cu).
// Diagnostic: AVD_STAGE_TIMES=1 brackets every stage of the tensor-core learn step with CUDA events and prints the durations
// at real clocks (ncu's per-launch times are taken with idle clocks and cold caches).  Synchronises: never set it in a bench.
struct StageTimer {
    bool on;
    cudaStream_t st;
    int n = 0;
    const char* names[32];
    cudaEvent_t ev[32];
    explicit StageTimer(cudaStream_t s) : st(s) {
        static const bool enabled = getenv("AVD_STAGE_TIMES") != nullptr;
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        cudaStreamIsCapturing(s, &cs);
        on = enabled && cs == cudaStreamCaptureStatusNone;
        mark("start");
    }
    void mark(const char* name) {
        if (!on || n >= 32) return;
        cudaEventCreate(&ev[n]);
        cudaEventRecord(ev[n], st);
        names[n++] = name;
    }
    ~StageTimer() {
        if (!on || n == 0) return;
        cudaEventSynchronize(ev[n - 1]);
        float total = 0.f;
        cudaEventElapsedTime(&total, ev[0], ev[n - 1]);
        fprintf(stderr, "[avd stage times] total %.1f us:", total * 1e3f);
        for (int i = 1; i < n; ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
            fprintf(stderr, " %s=%.1f", names[i], ms * 1e3f);
        }
        fprintf(stderr, "\n");
        for (int i = 0; i < n; ++i) cudaEventDestroy(ev[i]);
    }
};

// The preparation launch of the tensor-core learn step: weight half (V table, BN-folded 16-bit packs + folded biases of the four
// networks) and / or batch half (hi/lo-split [x_hi | 1 | x_lo] operand of the dgrad kernels).
static int learn_prep(const avd_learn_io* io, const Pass& p, const Workspace& w, int job_lo, int job_hi, bool vtab, bool batch, cudaStream_t st) {
    const avd_net_dims d = io->dims;
    const int A = io->A;
    const int64_t R = io->rows_per_agent, N = (int64_t)A * R;
    const CriticOff co = critic_off(d);
    const int64_t srs = io->s_stride ? io->s_stride : d.ns;
    const float* const prm[4] = {io->t_actor, io->t_critic, io->critic, io->actor};
    const bool crit[4] = {false, true, true, false};
    bf16* const W2b[4] = {nullptr, nullptr, w.cW2b, w.aW2b};
    bf16* const W2T[4] = {w.taW2T, w.tcW2T, w.cW2T, w.aW2T};
    float* const b2f[4] = {w.ta_b2f, w.tc_b2f, w.c_b2f, w.a_b2f};
    float* const wsc[4] = {nullptr, nullptr, w.wscale, w.wscale + A};
    PrepArgs pa = {};
    int Fmax = 0;
    AVD_TRY(p.pack_fold4(pa.jobs, Fmax, 4, prm, crit, W2b, W2T, b2f, wsc));
    pa.A = A; pa.l2 = d.l2; pa.f16 = p.f16() ? 1 : 0;
    // fold jobs [job_lo, job_hi) of {target actor, target critic, critic, actor}: z index of the fold grid = job * A + agent
    pa.fold_gx = (unsigned)((d.l2 + 31) / 32); pa.fold_gy = (unsigned)((Fmax + 7) / 8); pa.n_fold = pa.fold_gx * pa.fold_gy * (unsigned)((job_hi - job_lo) * A);
    pa.fold_z0 = (unsigned)(job_lo * A);
    pa.vtab_gy = (unsigned)((d.l2 + 31) / 32); pa.n_vtab = vtab ? (unsigned)A * pa.vtab_gy : 0u;
    pa.critic = io->critic; pa.cstride = co.total; pa.co = co; pa.d = d; pa.vtab = w.vtab;
    pa.v_rows = fused3::vtab_rows(); pa.v_stride = fused3::vtab_stride(); pa.v_total = fused3::vtab_floats();
    pa.s = io->s; pa.s_rs = srs; pa.a = io->a; pa.N = N; pa.xextT = w.xextT; pa.R = R; pa.Rp = (R + 63) / 64 * 64;
    const unsigned n_xext = batch ? (unsigned)((N + 255) / 256) : 0u;
    if (pa.n_vtab + pa.n_fold + n_xext == 0) return AVD_OK;
    learn_prep_kernel<<<pa.n_vtab + pa.n_fold + n_xext, 256, 0, st>>>(pa);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

// Side stream of the learn step (created on first use): the critic's unfold kernel -- 1216 small CTAs that need the gradients of
// BOTH critic products but feed nothing before the optimiser -- runs there while the actor's forward pass occupies the tensor pipe on
// the caller's stream (a 128-thread unfold CTA fits beside a persistent 220 KB CTA on the same SM).  Fork / join by events, so a
// CUDA-graph capture of the caller's stream records the branch.  Every caller shares the first side stream, except that a side stream
// joined into one capture stays in it until that capture ends: a caller that captures while it is so taken (the bodies of a
// conditional graph are captured concurrently) takes another idle one, or one created for it; with none, it runs unbranched.
struct SideStream {
    cudaStream_t caller = nullptr;
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr, fork2 = nullptr, join2 = nullptr, fork0 = nullptr, join0 = nullptr;
};
static bool side_idle(const SideStream& x) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(x.s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone;
}
static SideStream* side_stream(cudaStream_t caller) {
    constexpr int kSlots = 8;
    static SideStream tab[64][kSlots];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    SideStream* t = tab[dev];
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(caller, &cs) != cudaSuccess) return nullptr;
    const bool capturing = cs != cudaStreamCaptureStatusNone;
    int n = 0;
    while (n < kSlots && t[n].s) ++n;
    if (n > 0 && !capturing) return &t[0];
    for (int k = 0; k < n; ++k)
        if (t[k].caller == caller || side_idle(t[k])) return &t[k];
    // the first side stream is created outside a capture; further ones only for a capturing caller that found none idle
    if (n == kSlots || (n == 0 && capturing)) return nullptr;
    SideStream& x = t[n];
    if (cudaStreamCreateWithFlags(&x.s, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreateWithFlags(&x.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&x.join, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&x.fork2, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&x.join2, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&x.fork0, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&x.join0, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        x.s = nullptr;
        return nullptr;
    }
    x.caller = caller;
    return &x;
}

static int learn_fused3(const avd_learn_io* io, const Pass& p, const Workspace& w, cudaStream_t st) {
    StageTimer tm(st);
    static const bool no_side = getenv("AVD_NO_SIDE_STREAM") != nullptr || getenv("AVD_STAGE_TIMES") != nullptr;
    SideStream* side = no_side ? nullptr : side_stream(st);
    const avd_net_dims d = io->dims;
    const int A = io->A;
    const int64_t R = io->rows_per_agent, N = (int64_t)A * R;
    const ActorOff ao = actor_off(d);
    const CriticOff co = critic_off(d);
    const int F = d.l1 + d.la;
    constexpr int Fp = Workspace::kFp, MW = Workspace::kMaskWords;
    bf16* DZ = reinterpret_cast<bf16*>(w.DZ);
    float* Uc = w.U;
    float* Ua = w.U + (int64_t)A * d.l2;
    const bool f16 = p.f16();
    const int64_t srs = io->s_stride ? io->s_stride : d.ns;      // row pitch of the state batches
    float* const ws_c = w.wscale;
    float* const ws_a = w.wscale + A;
    // c_b2f .. ta_b2f (folded biases, written by the fold job), then dbm, ticket, U and sdq are adjacent in the workspace: one
    // memset zeroes every accumulator of the step.  (Running the weight half of the preparation on a side stream beside the
    // environment step and the replay gather was measured: -15 us per step with eager launches, nothing under CUDA-graph replay.)
    AVD_CUDA_OK(cudaMemsetAsync(w.c_b2f, 0, (size_t)((char*)(w.sdq + 2 * A) - (char*)w.c_b2f), st));
    // (only the target actor's pack is needed at once; running the rest of the preparation on the side stream beside the first pass was
    // measured: +9 us -- the 2400 small CTAs of the fold job get in the way of the persistent pass instead of hiding behind it)
    AVD_TRY(learn_prep(io, p, w, 0, 4, true, true, st));
    // fp16 backward tiles: dq ~ (q - y) / R (critic) and ~ dq/da / R (actor) are lifted by powers of two into the normal range of
    // fp16 (they saturate at +-65504 * 2^-k instead of overflowing); the unfold kernel divides the factors out again
    const float dm_c = f16 ? exp2f(ceilf(log2f((float)R))) : 1.0f, dm_a = f16 ? 256.0f * dm_c : 1.0f;
    AVD_LAUNCH_OK();
    tm.mark("fold+xext");
    // ---- TD target: y = r + gamma * target_critic(s', target_actor(s'))            trainer.py:493-494
    {
        fused3::RunArgs f = p.fused_args(fused3::MODE_ACTOR_OUT, io->t_actor, w.taW2T, w.ta_b2f, io->s2, srs);
        f.high = io->action_high; f.out = w.a2;
        AVD_TRY(fused3::run(f, st));
    }
    tm.mark("t_actor");
    {
        fused3::RunArgs f = p.fused_args(fused3::MODE_TARGET, io->t_critic, w.tcW2T, w.tc_b2f, io->s2, srs);
        f.act = w.a2; f.rew = io->r; f.gamma = io->gamma; f.hp = io->agent_hp; f.out = w.y;
        AVD_TRY(fused3::run(f, st));
    }
    tm.mark("t_critic");
    const int ncta = ctas_per_agent(A, R);
    const int64_t g2_cta = (int64_t)Workspace::kG2Rows * d.l2, g2_agent = (int64_t)ncta * g2_cta;
    float* const dbm_a = w.dbm + (int64_t)A * d.l2;
    // The actor's chain needs the critic's WEIGHTS, not its gradients, so its first half goes in front of the critic's backward pass: the
    // elementwise kernel that forms the actor's backward tile (HBM-bound, 55 us) then runs on the side stream beside the critic's
    // backward pass (tensor-bound), and the critic's unfold beside the actor's dgrad.  Both chains have their own tile / mask / slice buffers.
    // ---- actor loss gradient, first half: pi(s), d(-mean q)/d pi                    trainer.py:501-506
    {   // pi, the sign masks and d(action)/d(pre-activation) for the backward
        fused3::RunArgs f = p.fused_args(fused3::MODE_ACTOR_SAVE, io->actor, w.aW2T, w.a_b2f, io->s, srs);
        f.high = io->action_high; f.out = w.a2; f.mask_out = w.mask_a; f.mask2_out = w.mask2; f.dact_out = w.dact;
        AVD_TRY(fused3::run(f, st));
    }
    tm.mark("actor_fwd");
    {   // d(-mean q)/d pi
        fused3::RunArgs f = p.fused_args(fused3::MODE_CRITIC_ACTION, io->critic, w.cW2T, w.c_b2f, io->s, srs);
        f.act = w.a2; f.vtab = w.vtab; f.out = w.dpi; f.loss = io->loss;
        AVD_TRY(fused3::run(f, st));
    }
    tm.mark("critic_action");
    {
        cudaStream_t sd = st;
        if (side) {    // branch A: the actor's backward tile beside the critic's backward pass
            AVD_CUDA_OK(cudaEventRecord(side->fork, st));
            AVD_CUDA_OK(cudaStreamWaitEvent(side->s, side->fork, 0));
            sd = side->s;
        }
        const dim3 grid((unsigned)std::min<int64_t>((R + 15) / 16, std::max(1, 8 * sm_count() / A)), (unsigned)A);
        if (f16) AVD_CUDA_OK(launch_pdl(actor_dm_kernel<true>, grid, dim3(256), 0, sd, (const float*)w.dpi, (const float*)w.dact, (const uint32_t*)w.mask2, w.DZa, w.sdq + A, R, dm_a));
        else AVD_CUDA_OK(launch_pdl(actor_dm_kernel<false>, grid, dim3(256), 0, sd, (const float*)w.dpi, (const float*)w.dact, (const uint32_t*)w.mask2, w.DZa, w.sdq + A, R, dm_a));
        AVD_LAUNCH_OK();
        if (side) AVD_CUDA_OK(cudaEventRecord(side->join, side->s));
    }
    tm.mark("actor_bwd");
    // ---- critic loss gradient on (s, a)                                             trainer.py:495-498
    {
        fused3::RunArgs f = p.fused_args(fused3::MODE_CRITIC_BWD, io->critic, w.cW2T, w.c_b2f, io->s, srs);
        f.act = io->a; f.y = w.y; f.out = w.q; f.mask_out = w.mask; f.DZ_out = DZ; f.dm_scale = dm_c; f.sdq = w.sdq; f.loss = io->loss;
        AVD_TRY(fused3::run(f, st));
    }
    tm.mark("critic_bwd");
    // dgrad first, wgrad second: the unfold kernel then finds the 23 MB of partial G2 slices the weight-gradient CTAs have just written
    // still in L2 (after a dgrad pass, which streams 340 MB, it read them back from HBM)
    AVD_TRY(p.dgrad3_only(DZ, w.cW2b, F, Fp, w.mask, MW, w.xextT, w.G1, w.dbm));
    tm.mark("critic_dgrad");
    AVD_TRY(wgrad3::run(f16, d, true, A, R, io->critic, co.total, io->s, srs, io->a, DZ, w.G2part, g2_agent, g2_cta, st));
    tm.mark("critic_wgrad");
    if (side) {        // branch B: the critic's unfold beside the actor's dgrad
        AVD_CUDA_OK(cudaEventRecord(side->fork2, st));
        AVD_CUDA_OK(cudaStreamWaitEvent(side->s, side->fork2, 0));
        Pass ps = p;
        ps.st = side->s;
        AVD_TRY(ps.unfold(true, io->critic, F, Fp, w.G1, w.G2part, io->critic_grad, w.dbm, w.c_b2f, Uc, w.sdq, w.ticket, ws_c, dm_c));
        AVD_CUDA_OK(cudaEventRecord(side->join2, side->s));
    } else {
        AVD_TRY(p.unfold(true, io->critic, F, Fp, w.G1, w.G2part, io->critic_grad, w.dbm, w.c_b2f, Uc, w.sdq, w.ticket, ws_c, dm_c));
    }
    tm.mark("critic_unfold");
    // ---- actor loss gradient, second half
    if (side) AVD_CUDA_OK(cudaStreamWaitEvent(st, side->join, 0));      // join A: the actor's backward tile is complete
    AVD_TRY(p.dgrad3_only(w.DZa, w.aW2b, d.l1, Fp, w.mask_a, 8, w.xextT, w.G1a, dbm_a));
    tm.mark("actor_dgrad");
    AVD_TRY(wgrad3::run(f16, d, false, A, R, io->actor, ao.total, io->s, srs, nullptr, w.DZa, w.G2part_a, g2_agent, g2_cta, st));
    tm.mark("actor_wgrad");
    AVD_TRY(p.unfold(false, io->actor, d.l1, Fp, w.G1a, w.G2part_a, io->actor_grad, dbm_a, w.a_b2f, Ua, w.sdq + A, w.ticket + A, ws_a, dm_a));
    tm.mark("actor_unfold");
    if (side) AVD_CUDA_OK(cudaStreamWaitEvent(st, side->join2, 0));      // join B: the critic's gradients are complete
    const int rc = apply_local_updates(io, (void*)st);
    tm.mark("adam+polyak");
    return rc;
}

extern "C" int avd_ddpg_learn(const avd_learn_io* io, void* stream) {
    AVD_REQUIRE(io, "null io");
    AVD_TRY(check_dims(&io->dims, io->precision));
    AVD_REQUIRE(io->s && io->a && io->r && io->s2, "null batch");
    AVD_REQUIRE(io->actor && io->critic && io->t_actor && io->t_critic && io->actor_grad && io->critic_grad, "null parameters");
    AVD_REQUIRE(io->A >= 0 && io->rows_per_agent >= 1, "bad sizes");
    AVD_REQUIRE(!io->apply_updates || (io->actor_m && io->actor_v && io->critic_m && io->critic_v && io->actor_t && io->critic_t),
                "apply_updates needs Adam state");
    const avd_net_dims d = io->dims;
    const int A = io->A;
    const int64_t R = io->rows_per_agent, N = (int64_t)A * R;
    AVD_REQUIRE(io->workspace && io->workspace_bytes >= avd_ddpg_workspace_bytes(&d, A, R, io->precision), "workspace too small");
    if (A == 0) return AVD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const bool tc = io->precision != 0;
    const Pass p{d, A, io->precision, R, st};
    const ActorOff ao = actor_off(d);
    const CriticOff co = critic_off(d);
    const int F = d.l1 + d.la;
    Workspace w;
    const bool fz = fused_path(d, io->precision);   // persistent fused pass / dgrad / wgrad kernels
    w.carve(io->workspace, d, A, N, fz, operand_planes(io->precision));
    const dim3 gl1b((unsigned)((R + kL1BwdRows - 1) / kL1BwdRows), A);
    const int64_t srs = io->s_stride ? io->s_stride : d.ns;      // row pitch of the state batches
    AVD_REQUIRE(srs >= d.ns, "s_stride %d is smaller than the state width %d", (int)io->s_stride, d.ns);

    AVD_CUDA_OK(cudaMemsetAsync(io->actor_grad, 0, (size_t)A * ao.n_train * sizeof(float), st));
    AVD_CUDA_OK(cudaMemsetAsync(io->critic_grad, 0, (size_t)A * co.n_train * sizeof(float), st));
    if (io->loss) AVD_CUDA_OK(cudaMemsetAsync(io->loss, 0, (size_t)A * 2 * sizeof(float), st));
    if (fz) return learn_fused3(io, p, w, st);
    if (tc) {   // 16-bit copies (precision 3: split planes) of the four layer-2 kernels (K-major for forward, and for dgrad on the online nets)
        AVD_TRY(p.pack(io->t_actor, ao.total, ao.W2, d.l1, nullptr, w.taW2T));
        AVD_TRY(p.pack(io->t_critic, co.total, co.W2, F, nullptr, w.tcW2T));
        AVD_TRY(p.pack(io->critic, co.total, co.W2, F, w.cW2b, w.cW2T));
        AVD_TRY(p.pack(io->actor, ao.total, ao.W2, d.l1, w.aW2b, w.aW2T));
    }
    // ---- TD target: y = r + gamma * target_critic(s', target_actor(s'))            trainer.py:493-494
    AVD_TRY(p.layer1(false, io->t_actor, io->s2, srs, 1, nullptr, w.H1a));
    AVD_TRY(p.forward(w.H1a, d.l1, io->t_actor, ao.total, ao.W2, w.taW2T, w.Z));
    {
        HeadArgs h = actor_head(d, io->t_actor, w.Z, R, io->action_high);
        h.out = w.a2;
        AVD_TRY(launch_head<HEAD_ACTOR_FWD>(h, d.l2, A, st));
    }
    AVD_TRY(p.layer1(true, io->t_critic, io->s2, srs, 1, w.a2, w.H));
    AVD_TRY(p.forward(w.H, F, io->t_critic, co.total, co.W2, w.tcW2T, w.Z));
    {
        HeadArgs h = critic_head(d, io->t_critic, w.Z, R);
        h.rew = io->r; h.gamma = io->gamma; h.hp = io->agent_hp; h.out = w.y;
        if (io->agent_hp) AVD_TRY(launch_head<HEAD_CRITIC_TARGET_HP>(h, d.l2, A, st));
        else AVD_TRY(launch_head<HEAD_CRITIC_TARGET>(h, d.l2, A, st));
    }
    // ---- critic loss gradient on (s, a)                                             trainer.py:495-498
    AVD_TRY(p.layer1(true, io->critic, io->s, srs, 1, io->a, w.H));
    AVD_TRY(p.forward(w.H, F, io->critic, co.total, co.W2, w.cW2T, w.Z));
    {
        HeadArgs h = critic_head(d, io->critic, w.Z, R);
        h.y = w.y; h.out = w.q; h.DZ = w.DZ; h.grads = io->critic_grad; h.gstride = co.n_train; h.loss = io->loss;
        AVD_TRY(launch_head<HEAD_CRITIC_BWD>(h, d.l2, A, st, io->precision));
    }
    AVD_TRY(p.wgrad(w.H, F, w.DZ, io->critic_grad, co.n_train, co.W2));
    AVD_TRY(p.dgrad(w.DZ, io->critic, co.total, co.W2, w.cW2b, F, 0, F, w.DH));
    l1_backward_kernel<true><<<gl1b, 128, 0, st>>>(d, io->critic, co.total, io->s, srs, io->a, R, w.DH, io->critic_grad, co.n_train);
    AVD_LAUNCH_OK();
    // ---- actor loss gradient: -mean(critic(s, actor(s)))                            trainer.py:501-506
    AVD_TRY(p.layer1(false, io->actor, io->s, srs, 1, nullptr, w.H1a));
    AVD_TRY(p.forward(w.H1a, d.l1, io->actor, ao.total, ao.W2, w.aW2T, w.Za));
    {
        HeadArgs h = actor_head(d, io->actor, w.Za, R, io->action_high);
        h.out = w.a2;   // pi
        AVD_TRY(launch_head<HEAD_ACTOR_FWD>(h, d.l2, A, st));
    }
    AVD_TRY(p.layer1(true, io->critic, io->s, srs, 1, w.a2, w.H));
    AVD_TRY(p.forward(w.H, F, io->critic, co.total, co.W2, w.cW2T, w.Z));
    {
        HeadArgs h = critic_head(d, io->critic, w.Z, R);
        h.DZ = w.DZ; h.loss = io->loss;
        AVD_TRY(launch_head<HEAD_CRITIC_BWD_ACTION>(h, d.l2, A, st, io->precision));
    }
    AVD_TRY(p.dgrad(w.DZ, io->critic, co.total, co.W2, w.cW2b, F, d.l1, d.la, w.DH));   // action columns only
    action_grad_kernel<<<dim3((unsigned)std::min<int64_t>((R + 255) / 256, 2048), A), 256, 0, st>>>(d, io->critic, co.total, w.a2, R, w.DH, w.dpi);
    AVD_LAUNCH_OK();
    {
        HeadArgs h = actor_head(d, io->actor, w.Za, R, io->action_high);
        h.dpi = w.dpi; h.DZ = w.DZ; h.grads = io->actor_grad; h.gstride = ao.n_train;
        AVD_TRY(launch_head<HEAD_ACTOR_BWD>(h, d.l2, A, st, io->precision));
    }
    AVD_TRY(p.wgrad(w.H1a, d.l1, w.DZ, io->actor_grad, ao.n_train, ao.W2));
    AVD_TRY(p.dgrad(w.DZ, io->actor, ao.total, ao.W2, w.aW2b, d.l1, 0, d.l1, w.DH));
    l1_backward_kernel<false><<<gl1b, 128, 0, st>>>(d, io->actor, ao.total, io->s, srs, nullptr, R, w.DH, io->actor_grad, ao.n_train);
    AVD_LAUNCH_OK();
    return apply_local_updates(io, stream);
}

