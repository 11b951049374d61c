// avd_replay.cu -- GPU-resident replay rings (src/replaybuffer.py) for all M*P agents at once.
//
// Ring r = m*P + p lives at ring[slot][r][10]: one 40-byte record (s[4], a, r, s'[4]) per agent and slot,
// so ReplayBuffer.add for the whole population is one coalesced sweep over a slot (fused into
// avd_env_step; avd_replay_add is the stand-alone form) and a sampled record costs two 32-byte sectors.
// Index draws replace np.random.choice (replaybuffer.py:54) by Philox words mapped with a 64-bit
// multiply-shift, bit-exact against oracle/philox_np.py:replay_indices.
#include "avd_common.cuh"
#include "avd_rng.cuh"

namespace avd {

__global__ void __launch_bounds__(256) replay_add_kernel(float* __restrict__ ring, int64_t capacity, int64_t n_rings,
                                                         const avd_clock* __restrict__ clock, const float* __restrict__ s,
                                                         const float* __restrict__ a, const float* __restrict__ r,
                                                         const float* __restrict__ s2) {
    const int64_t slot = (int64_t)(clock->ring_count % (uint64_t)capacity);   // replaybuffer.py:40
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_rings; v += (int64_t)gridDim.x * blockDim.x) {
        float2* rec = reinterpret_cast<float2*>(ring + (slot * n_rings + v) * AVD_RING_RECORD_FLOATS);
        rec[0] = make_float2(s[v], s[n_rings + v]);
        rec[1] = make_float2(s[2 * n_rings + v], s[3 * n_rings + v]);
        rec[2] = make_float2(a[v], r[v]);
        rec[3] = make_float2(s2[v], s2[n_rings + v]);
        rec[4] = make_float2(s2[2 * n_rings + v], s2[3 * n_rings + v]);
    }
}

// RUNS: every ring's stream is keyed by its run (ring_key); a separate instantiation so the one-run kernels keep their code.
template <bool RUNS>
__global__ void __launch_bounds__(256) replay_indices_kernel(int64_t* __restrict__ idx_out, int64_t n_rings, int64_t ring_id_base,
                                                             int32_t batch, int64_t capacity, uint64_t seed,
                                                             const avd_clock* __restrict__ clock, const __grid_constant__ avd_runs rt) {
    const uint64_t count = clock->ring_count;
    const uint64_t range = count < (uint64_t)capacity ? count : (uint64_t)capacity;   // replaybuffer.py:52
    const uint32_t tick = (uint32_t)clock->update_tick;
    const int64_t blocks_per_ring = batch / 4;
    const int64_t total = n_rings * blocks_per_ring;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ring = t / blocks_per_ring, jb = t - ring * blocks_per_ring;
        const StreamKey key = ring_key(RUNS ? &rt : nullptr, seed, (uint64_t)(ring_id_base + ring));
        const uint64_t id = key.id * (uint64_t)blocks_per_ring + (uint64_t)jb;
        const uint4 w = rng_words(key.seed, id, tick, AVD_RNG_REPLAY);
        longlong4* dst = reinterpret_cast<longlong4*>(idx_out + ring * batch + jb * 4);
        *dst = make_longlong4(index_from_word(w.x, range), index_from_word(w.y, range), index_from_word(w.z, range),
                              index_from_word(w.w, range));
    }
}

__global__ void __launch_bounds__(256) replay_gather_kernel(const float* __restrict__ ring, int64_t n_rings,
                                                            const int64_t* __restrict__ idx, int32_t batch,
                                                            float* __restrict__ s, float* __restrict__ a, float* __restrict__ r,
                                                            float* __restrict__ s2) {
    const int64_t total = n_rings * batch;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < total; n += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ringid = n / batch;
        const int64_t slot = idx[n];
        const float2* rec = reinterpret_cast<const float2*>(ring + (slot * n_rings + ringid) * AVD_RING_RECORD_FLOATS);
        const float2 q0 = __ldg(rec), q1 = __ldg(rec + 1), q2 = __ldg(rec + 2), q3 = __ldg(rec + 3), q4 = __ldg(rec + 4);
        reinterpret_cast<float4*>(s)[n] = make_float4(q0.x, q0.y, q1.x, q1.y);
        a[n] = q2.x;
        r[n] = q2.y;
        reinterpret_cast<float4*>(s2)[n] = make_float4(q3.x, q3.y, q4.x, q4.y);
    }
}

// index draw + gather fused: thread t owns Philox block jb of ring `ring` (four samples).  All four records (20 x 8 bytes) are requested
// before the first use, so a thread overlaps four TLB / DRAM latencies instead of one; outputs are 16-byte stores.
template <bool RUNS>
__global__ void __launch_bounds__(256) replay_sample_kernel(const float* __restrict__ ring, int64_t n_rings, int64_t ring_id_base, int32_t batch,
                                                            int64_t capacity, uint64_t seed, const avd_clock* __restrict__ clock,
                                                            int64_t* __restrict__ idx_out, float* __restrict__ s, float* __restrict__ a,
                                                            float* __restrict__ r, float* __restrict__ s2, const __grid_constant__ avd_runs rt) {
    const uint64_t count = clock->ring_count;
    const uint64_t range = count < (uint64_t)capacity ? count : (uint64_t)capacity;   // replaybuffer.py:52
    const uint32_t tick = (uint32_t)clock->update_tick;
    const int64_t blocks_per_ring = batch / 4;
    const int64_t total = n_rings * blocks_per_ring;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t rg = t / blocks_per_ring, jb = t - rg * blocks_per_ring;
        const StreamKey key = ring_key(RUNS ? &rt : nullptr, seed, (uint64_t)(ring_id_base + rg));
        const uint64_t id = key.id * (uint64_t)blocks_per_ring + (uint64_t)jb;
        const uint4 w = rng_words(key.seed, id, tick, AVD_RNG_REPLAY);
        const int64_t ix[4] = {index_from_word(w.x, range), index_from_word(w.y, range), index_from_word(w.z, range), index_from_word(w.w, range)};
        const int64_t n0 = rg * batch + jb * 4;
        if (idx_out) *reinterpret_cast<longlong4*>(idx_out + n0) = make_longlong4(ix[0], ix[1], ix[2], ix[3]);
        float2 q[4][5];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float2* rec = reinterpret_cast<const float2*>(ring + (ix[u] * n_rings + rg) * AVD_RING_RECORD_FLOATS);
#pragma unroll
            for (int k = 0; k < 5; ++k) q[u][k] = __ldg(rec + k);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            reinterpret_cast<float4*>(s)[n0 + u] = make_float4(q[u][0].x, q[u][0].y, q[u][1].x, q[u][1].y);
            reinterpret_cast<float4*>(s2)[n0 + u] = make_float4(q[u][3].x, q[u][3].y, q[u][4].x, q[u][4].y);
        }
        *reinterpret_cast<float4*>(a + n0) = make_float4(q[0][2].x, q[1][2].x, q[2][2].x, q[3][2].x);
        *reinterpret_cast<float4*>(r + n0) = make_float4(q[0][2].y, q[1][2].y, q[2][2].y, q[3][2].y);
    }
}

__global__ void __launch_bounds__(256) replay_fill_kernel(float* __restrict__ ring, int64_t n_records, uint64_t seed) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_records; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 w0 = rng_words(seed, (uint64_t)i, 0u, 0x7F);
        const uint4 w1 = rng_words(seed, (uint64_t)i, 1u, 0x7F);
        const float e0 = uniform_sym(w0.x, 4.0f), e1 = uniform_sym(w0.y, 4.0f), a0 = uniform_sym(w0.z, 1.0f), al = uniform_sym(w0.w, 1.0f);
        const float u = uniform_sym(w1.x, 2.5f);
        const float rew = -(0.02f * fabsf(e0) + 0.01f * fabsf(e1) + 0.08f * fabsf(u));
        float2* rec = reinterpret_cast<float2*>(ring + i * AVD_RING_RECORD_FLOATS);
        rec[0] = make_float2(e0, e1);
        rec[1] = make_float2(a0, al);
        rec[2] = make_float2(u, rew);
        rec[3] = make_float2(e0 + 0.1f * e1 - 0.1f * a0, e1 - 0.1f * a0 + 0.1f * al);
        rec[4] = make_float2(u, uniform_sym(w1.y, 1.0f));
    }
}

__global__ void rng_words_kernel(uint32_t* __restrict__ out, int64_t n, uint64_t id_base, uint32_t tick, uint32_t purpose, uint64_t seed) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        reinterpret_cast<uint4*>(out)[i] = rng_words(seed, id_base + (uint64_t)i, tick, purpose);
    }
}

__global__ void rng_normals_kernel(float* __restrict__ out, int64_t n, uint64_t id_base, uint32_t tick, uint32_t purpose, uint64_t seed) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 w = rng_words(seed, id_base + (uint64_t)i, tick, purpose);
        float z0, z1, z2, z3;
        normal_pair(w.x, w.y, z0, z1);
        normal_pair(w.z, w.w, z2, z3);
        reinterpret_cast<float4*>(out)[i] = make_float4(z0, z1, z2, z3);
    }
}

}  // namespace avd

using namespace avd;

extern "C" int avd_replay_add(float* ring, int64_t capacity, int64_t M, int64_t P, const avd_clock* clock, const float* s,
                              const float* a, const float* r, const float* s2, void* stream) {
    AVD_REQUIRE(ring && clock && s && a && r && s2, "null buffer");
    AVD_REQUIRE(capacity > 0 && M > 0 && P >= 0, "bad sizes");
    if (P == 0) return AVD_OK;
    replay_add_kernel<<<grid_for(M * P), 256, 0, (cudaStream_t)stream>>>(ring, capacity, M * P, clock, s, a, r, s2);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

static int replay_sample_indices(int64_t* idx_out, int64_t n_rings, int64_t ring_id_base, int32_t batch, int64_t capacity, uint64_t seed,
                                 const avd_runs* runs, const avd_clock* clock, void* stream) {
    AVD_REQUIRE(idx_out && clock, "null buffer");
    AVD_REQUIRE(batch > 0 && batch % 4 == 0, "batch must be a positive multiple of 4 (got %d)", batch);
    AVD_REQUIRE(capacity > 0 && n_rings >= 0, "bad sizes");
    if (n_rings == 0) return AVD_OK;
    if (runs)
        replay_indices_kernel<true><<<grid_for(n_rings * (batch / 4)), 256, 0, (cudaStream_t)stream>>>(idx_out, n_rings, 0, batch, capacity, 0,
                                                                                                       clock, *runs);
    else
        replay_indices_kernel<false><<<grid_for(n_rings * (batch / 4)), 256, 0, (cudaStream_t)stream>>>(idx_out, n_rings, ring_id_base, batch,
                                                                                                        capacity, seed, clock, avd_runs{});
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_replay_sample_indices(int64_t* idx_out, int64_t n_rings, int64_t ring_id_base, int32_t batch,
                                         int64_t capacity, uint64_t seed, const avd_clock* clock, void* stream) {
    return replay_sample_indices(idx_out, n_rings, ring_id_base, batch, capacity, seed, nullptr, clock, stream);
}

extern "C" int avd_replay_sample_indices_runs(int64_t* idx_out, int64_t n_rings, int32_t batch, int64_t capacity, const avd_runs* runs,
                                              const avd_clock* clock, void* stream) {
    AVD_REQUIRE(runs, "null run table");
    AVD_REQUIRE(runs->seed && runs->runs >= 1 && runs->platoons_per_run >= 1 &&
                    n_rings % ((int64_t)runs->runs * runs->platoons_per_run) == 0,
                "%lld rings are not M x (%d runs x %lld platoons), or the table has no seeds", (long long)n_rings, (int)runs->runs,
                (long long)runs->platoons_per_run);
    return replay_sample_indices(idx_out, n_rings, 0, batch, capacity, 0, runs, clock, stream);
}

extern "C" int avd_replay_gather(const float* ring, int64_t capacity, int64_t M, int64_t P, const int64_t* idx, int32_t batch,
                                 float* s, float* a, float* r, float* s2, void* stream) {
    AVD_REQUIRE(ring && idx && s && a && r && s2, "null buffer");
    AVD_REQUIRE(capacity > 0 && M > 0 && P >= 0 && batch > 0, "bad sizes");
    if (P == 0) return AVD_OK;
    replay_gather_kernel<<<grid_for(M * P * batch), 256, 0, (cudaStream_t)stream>>>(ring, M * P, idx, batch, s, a, r, s2);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

static int replay_sample(const float* ring, int64_t capacity, int64_t M, int64_t P, int64_t ring_id_base, int32_t batch, uint64_t seed,
                         const avd_runs* runs, const avd_clock* clock, int64_t* idx_out, float* s, float* a, float* r, float* s2, void* stream) {
    AVD_REQUIRE(ring && clock && s && a && r && s2, "null buffer");
    AVD_REQUIRE(batch > 0 && batch % 4 == 0, "batch must be a positive multiple of 4 (got %d)", batch);
    AVD_REQUIRE(capacity > 0 && M > 0 && P >= 0, "bad sizes");
    AVD_REQUIRE(((uintptr_t)a & 15) == 0 && ((uintptr_t)r & 15) == 0 && ((uintptr_t)s & 15) == 0 && ((uintptr_t)s2 & 15) == 0 &&
                (!idx_out || ((uintptr_t)idx_out & 31) == 0), "sample outputs must be 16-byte (indices: 32-byte) aligned");
    if (P == 0) return AVD_OK;
    if (runs)
        replay_sample_kernel<true><<<grid_for(M * P * (batch / 4)), 256, 0, (cudaStream_t)stream>>>(ring, M * P, 0, batch, capacity, 0, clock, idx_out, s,
                                                                                                    a, r, s2, *runs);
    else
        replay_sample_kernel<false><<<grid_for(M * P * (batch / 4)), 256, 0, (cudaStream_t)stream>>>(ring, M * P, ring_id_base, batch, capacity, seed, clock,
                                                                                                     idx_out, s, a, r, s2, avd_runs{});
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_replay_sample(const float* ring, int64_t capacity, int64_t M, int64_t P, int64_t ring_id_base, int32_t batch, uint64_t seed,
                                 const avd_clock* clock, int64_t* idx_out, float* s, float* a, float* r, float* s2, void* stream) {
    return replay_sample(ring, capacity, M, P, ring_id_base, batch, seed, nullptr, clock, idx_out, s, a, r, s2, stream);
}

extern "C" int avd_replay_sample_runs(const float* ring, int64_t capacity, int64_t M, int64_t P, int32_t batch, const avd_runs* runs,
                                      const avd_clock* clock, int64_t* idx_out, float* s, float* a, float* r, float* s2, void* stream) {
    AVD_REQUIRE(runs, "null run table");
    AVD_REQUIRE_RUNS(runs, P);
    return replay_sample(ring, capacity, M, P, 0, batch, 0, runs, clock, idx_out, s, a, r, s2, stream);
}

extern "C" int avd_replay_fill_synthetic(float* ring, int64_t capacity, int64_t M, int64_t P, uint64_t seed, void* stream) {
    AVD_REQUIRE(ring, "null ring");
    AVD_REQUIRE(capacity > 0 && M > 0 && P >= 0, "bad sizes");
    if (P == 0) return AVD_OK;
    replay_fill_kernel<<<grid_for(capacity * M * P), 256, 0, (cudaStream_t)stream>>>(ring, capacity * M * P, seed);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_rng_words(uint32_t* out4, int64_t n, uint64_t id_base, uint32_t tick, uint32_t purpose, uint64_t seed, void* stream) {
    AVD_REQUIRE(out4 && n >= 0, "bad args");
    if (n == 0) return AVD_OK;
    rng_words_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(out4, n, id_base, tick, purpose, seed);
    AVD_LAUNCH_OK();
    return AVD_OK;
}

extern "C" int avd_rng_normals(float* out4, int64_t n, uint64_t id_base, uint32_t tick, uint32_t purpose, uint64_t seed, void* stream) {
    AVD_REQUIRE(out4 && n >= 0, "bad args");
    if (n == 0) return AVD_OK;
    rng_normals_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(out4, n, id_base, tick, purpose, seed);
    AVD_LAUNCH_OK();
    return AVD_OK;
}
