// Shared definitions for the sm_100a gossip kernels.
//
// Data plane design (see DESIGN.md):
//   * every rank owns, in NVSwitch peer-mapped ("symmetric") memory,
//       - a signal pad  (SgpSignalPad): sequence flags + push-sum weight
//       - an outbox     (2 x n floats, double buffered by step parity)
//   * a gossip step is a PULL: the producer writes its outbox and releases a
//     per-CTA sequence flag; consumers acquire the flag over NVLink and read
//     the outbox with 16-byte P2P loads, applying the edge weight while they
//     accumulate.  Write-after-read on the outbox is fenced by a per-reader
//     ack sequence the consumer stores back into the producer's pad.
//   * the time-varying graph is a device table indexed by step % period.
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#define SGP_MAX_PEERS   8      // peers per iteration (== topology.MAX_PEERS_PER_ITR)
#define SGP_MAX_RANKS   64     // ranks in one NVLink domain
#define SGP_MAX_CTAS    1024   // upper bound on the (persistent) grid size
#define SGP_THREADS     256
#define SGP_VEC         4      // floats per 16-byte access
#define SGP_UNROLL      4      // 16-byte accesses in flight per thread
#define SGP_CHUNK       (SGP_THREADS * SGP_VEC * SGP_UNROLL)   // 4096 elements
#define SGP_TABLE_ROW   (2 + 2 * SGP_MAX_PEERS)                // n_in,n_out,in[8],out[8]
#define SGP_WTABLE_ROW  (1 + SGP_MAX_PEERS)                    // self_w, in_w[8]
#define SGP_SEQ_STRIDE  16     // pub_seq = step * 16 + segments_published  (<= 15 segments)

// status codes written to SgpState::status (0 == healthy)
#define SGP_OK               0
#define SGP_ERR_TIMEOUT_PUB  1   // in-neighbour never published (heartbeat)
#define SGP_ERR_TIMEOUT_ACK  2   // out-neighbour never released our outbox
#define SGP_ERR_TIMEOUT_BAR  3   // device barrier timed out

// ---- symmetric (peer-visible) per-rank signal pad --------------------------
struct __align__(128) SgpSignalPad {
    // pub_seq[b] == s*SGP_SEQ_STRIDE + k  <=>  the first k segments of CTA b's share of
    // outbox[s&1] for step s are visible (k == segments: all of it)
    uint32_t pub_seq[SGP_MAX_CTAS];
    // ack_seq[r] == s+1  <=>  rank r finished reading our outbox of step s
    uint32_t ack_seq[SGP_MAX_RANKS];
    // push-sum weight that belongs to outbox[parity]
    float    psw[2];
    uint32_t _pad0[30];
    // device barrier: bar_seq[r] is bumped by rank r
    uint32_t bar_seq[SGP_MAX_RANKS];
    // AD-PSGD bilateral handshake (round counters)
    uint32_t bilat_pub;      // rounds published by the owner
    uint32_t _pad1[31];
};

// ---- local (non-peer) per-rank kernel state --------------------------------
struct __align__(128) SgpState {
    uint32_t step;          // gossip steps completed (drives parity + phase)
    uint32_t done_ctas;     // CTAs finished in the current launch
    uint32_t status;        // SGP_ERR_* (sticky)
    uint32_t bar_epoch;     // device-barrier epochs completed
    float    ps_weight[2];  // W[step&1] is current; kernel writes W[(step+1)&1]
    float    res_weight;    // overlap: push-sum weight of the pending residual
    uint32_t phase_base;    // row offset added to step before % period
    uint32_t bilat_round;   // AD-PSGD rounds completed
    uint32_t bilat_done;    // last probe outcome (1 = partner has published)
    uint32_t ack_from;      // outbox WAR fence only applies to steps >= ack_from + 2
    // AD-PSGD device-side round state machine (sgp_bilat_decide_kernel + SGP_F_FROM_STATE)
    uint32_t bilat_cmd;        // SGP_F_* bits the next worker launch executes (0 = nothing to do)
    uint32_t bilat_published;  // 1: this rank's snapshot of the current round is in the outbox
    uint32_t bilat_budget;     // rounds this rank may still START before its next gradient arrives
    uint32_t bilat_enabled;    // 0: gossip disabled (an in-flight round still completes)
    // soft heartbeat: a wait that exceeds soft_timeout_us is COUNTED (and keeps waiting until the
    // hard timeout); the host logs "gossip round delayed, still waiting" -- the one-sided
    // analogue of the reference re-queueing an interrupted round (gossip/distributed.py:358-364)
    uint32_t soft_timeout_us;  // 0 = off
    uint32_t soft_timeouts;    // waits that went past the soft deadline (monotonic)
    // overlap: factor the pending residual is multiplied with when it is folded.  1 when a gather
    // KERNEL produced it (already weighted); the in-neighbour's edge weight when the residual is
    // the raw outbox copied by the DMA engines (sgp_gather_wait / cudaMemcpyAsync / sgp_gather_ack)
    float    res_scale;
    uint32_t _pad[14];
};

// ---- hyper-parameters (device resident so CUDA graphs can retarget them) ----
struct SgpHyper {
    float lr;
    float momentum;
    float weight_decay;
    float nesterov;      // 0 / 1
    float do_sgd;        // 0 / 1  (first overlap step has no gradient yet)
    float grad_scale;    // multiplies the gradient (1/nprocs, loss-scale^-1 ...)
    float _pad[2];
};

// kernel mode bits
#define SGP_F_SGD        (1u << 0)   // apply SGD-momentum before publishing
#define SGP_F_GRAD_BF16  (1u << 1)   // gradient buffer is bf16 (else fp32)
#define SGP_F_SHADOW     (1u << 2)   // also write a bf16 copy of the params
#define SGP_F_ZERO_GRAD  (1u << 3)   // clear the gradient after consuming it
#define SGP_F_PHASE1     (1u << 4)   // run the local/publish phase
#define SGP_F_PHASE2     (1u << 5)   // run the pull/mix phase
#define SGP_F_FOLD_RES   (1u << 6)   // overlap: fold the pending residual in
#define SGP_F_NO_ROTATE  (1u << 7)   // do not advance step (flush kernels)
#define SGP_F_PUBLISH    (1u << 8)   // write outbox + release flags
#define SGP_F_IN_NUMER   (1u << 9)   // z already holds the numerator x (external optimizer)
#define SGP_F_KEEP_Z     (1u << 10)  // phase 1 publishes a snapshot but leaves z untouched
#define SGP_F_SELF_FROM_Z (1u << 11) // phase 2 mixes the CURRENT z (not the published snapshot)
#define SGP_F_FROM_STATE (1u << 12)  // take the mode bits from SgpState::bilat_cmd (set by the decide kernel)

struct SgpArgs {
    // local buffers (length n, n % SGP_CHUNK == 0)
    float*               z;          // de-biased parameters (fp32 master)
    void*                g;          // gradient (fp32 / bf16) or null
    float*               g2;         // optional 2nd gradient buffer (fp32), added to g:
                                     //   bf16 grads of the bf16 compute weights + fp32 grads
                                     //   of the fp32 (BatchNorm) parameters, same layout
    float*               m;          // momentum or null
    __nv_bfloat16*       shadow;     // bf16 copy of z or null
    float*               residual;   // overlap residual or null
    // symmetric memory: device arrays of per-rank base pointers
    SgpSignalPad* const* pads;       // [world]
    float* const*        outboxes;   // [world], each 2*n floats
    // schedule
    const int*           table;      // [period][SGP_TABLE_ROW]
    const float*         wtable;     // [period][SGP_WTABLE_ROW]
    int                  period;
    // identity
    int                  rank;
    int                  world;
    long long            n;
    // state
    SgpState*            st;
    const SgpHyper*      hyper;
    unsigned long long   timeout_ns;
    unsigned int         flags;
    int                  segments;   // phase-1/phase-2 interleave granularity per CTA
};

#ifdef __CUDACC__
// ---- PTX helpers -----------------------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_relaxed_sys_f32(const float* p) {
    float v;
    asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys_f32(float* p, float v) {
    asm volatile("st.relaxed.sys.global.f32 [%0], %1;" :: "l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// streaming 16-byte load that does not allocate in L1 (peer data is read once;
// peer addresses bypass the local L2 by construction of the NVLink aperture)
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
// local streaming loads with an L2 evict-first policy: data consumed exactly
// once (z, g, m, residual) must not push the freshly published outbox -- which
// phase 2 re-reads -- out of the 126 MB L2.  (On sm_100a the `.L2::evict_first`
// qualifier is only legal on 32-byte loads, so 16-byte loads carry the policy
// as an explicit cache hint.)
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_evict_last_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ float4 ld_once_f4(const float4* p, uint64_t pol) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ uint2 ld_once_u2(const uint2* p, uint64_t pol) {
    uint2 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;"
                 : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_hint_f4(float4* p, float4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_f4(float4* p, float4 v) {
    asm volatile("st.global.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_u2(uint2* p, uint2 v) {
    asm volatile("st.global.v2.u32 [%0], {%1,%2};" :: "l"(p), "r"(v.x), "r"(v.y) : "memory");
}

__device__ __forceinline__ float4 bf16x4_to_f4(uint2 r) {
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&r.x);
    __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&r.y);
    float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ uint2 f4_to_bf16x4(float4 v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
    __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<uint32_t*>(&a);
    r.y = *reinterpret_cast<uint32_t*>(&b);
    return r;
}

// Spin until *flag >= want (sequence numbers, wrap-safe compare) or timeout.
// Returns false on timeout / pre-existing error.  Called by ONE thread.
__device__ __forceinline__ bool spin_wait_geq(const uint32_t* flag, uint32_t want,
                                              SgpState* st, unsigned long long timeout_ns,
                                              uint32_t err_code) {
    if ((int32_t)(ld_acquire_sys(flag) - want) >= 0) return true;
    const unsigned long long t0 = globaltimer_ns();
    const unsigned long long soft_ns = (unsigned long long)(*((volatile uint32_t*)&st->soft_timeout_us)) * 1000ull;
    bool soft_hit = false;
    uint32_t polls = 0;
    while (true) {
        if ((int32_t)(ld_acquire_sys(flag) - want) >= 0) return true;
        if ((++polls & 63u) == 0u) {
            if (*((volatile uint32_t*)&st->status) != SGP_OK) return false;
            const unsigned long long waited = globaltimer_ns() - t0;
            if (waited > timeout_ns) {
                atomicCAS(&st->status, (uint32_t)SGP_OK, err_code);
                return false;
            }
            if (soft_ns != 0ull && !soft_hit && waited > soft_ns) {
                soft_hit = true;                    // counted once per wait; keep waiting
                atomicAdd(&st->soft_timeouts, 1u);
            }
        }
        __nanosleep(64);
    }
}

#endif  // __CUDACC__

// launcher entry points (sgp_kernels.cu)
extern "C" {
cudaError_t sgp_launch_step(const SgpArgs* args, int grid, cudaStream_t stream);
cudaError_t sgp_launch_step_pipe(const SgpArgs* args, int grid, cudaStream_t stream);
int sgp_max_resident_ctas_pipe(int device);
cudaError_t sgp_launch_gather(const SgpArgs* args, int grid, int pub_grid, cudaStream_t stream);
cudaError_t sgp_launch_gather_tma(const SgpArgs* args, int grid, int pub_grid, cudaStream_t stream);
cudaError_t sgp_launch_probe(const SgpArgs* args, int pub_grid, uint32_t* host_flag,
                             cudaStream_t stream);
cudaError_t sgp_launch_gather_wait(const SgpArgs* args, int pub_grid, cudaStream_t stream);
cudaError_t sgp_launch_gather_ack(const SgpArgs* args, cudaStream_t stream);
cudaError_t sgp_launch_bilat_decide(const SgpArgs* args, int pub_grid, int passive,
                                    unsigned long long max_wait_ns, uint32_t* host_fb, cudaStream_t stream);
cudaError_t sgp_launch_bilat_ctl(SgpState* st, int budget, int enabled, cudaStream_t stream);
cudaError_t sgp_launch_zero(void* p, long long bytes, cudaStream_t stream);
cudaError_t sgp_launch_peer_reduce(float* dst, const float* const* srcs, int nsrc, long long n, float scale,
                                   cudaStream_t stream);
cudaError_t sgp_launch_scale(float* x, long long n, const float* scalar, int invert,
                             __nv_bfloat16* shadow, cudaStream_t stream);
cudaError_t sgp_launch_barrier(SgpSignalPad* const* pads, SgpState* st, int rank, int world,
                               unsigned long long timeout_ns, cudaStream_t stream);
cudaError_t sgp_launch_allreduce_sgd(const SgpArgs* args, void* const* grad_peers, int grid,
                                     cudaStream_t stream);
int sgp_max_resident_ctas(int device);
cudaError_t sgp_preload_kernels();
}
