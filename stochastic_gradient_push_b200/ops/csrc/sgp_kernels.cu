// sm_100a gossip kernels: fused SGD + push-sum mix over NVSwitch peer memory.
//
// Replaces, in ONE launch per training step, the reference's K1-K9 elementwise
// swarm (ps_numerator / unbias / residual add / pre-scale / flatten / scale /
// accumulate / unflatten / optimizer.step; gossip/distributed.py:298-455,
// gossip/gossiper.py:125-219, gossip_sgd.py:389) and its N1-N3 NCCL broadcasts.
//
//   sgp_step_kernel    phase 1: x = z*w ; SGD-momentum ; (+residual) ; publish
//                      phase 2: acquire in-neighbours' flags ; weighted P2P
//                               loads ; push-sum weight update ; de-bias ; store
//   sgp_gather_kernel  Overlap-SGP: residual = sum_k w_k * outbox_k  (side stream)
//   sgp_probe_kernel   AD-PSGD passive poll ("has my partner published?")
//   sgp_allreduce_sgd  AR-SGD comparator: one-shot P2P all-reduce fused with SGD
//   sgp_barrier_kernel device-side barrier over the signal pads
//   sgp_scale_kernel   flat x *= w  /  x /= w  (ps_numerator / unbias API parity)
#include <cuda.h>

#include "sgp_common.cuh"

namespace {

struct RowInfo {
    int   n_in, n_out;
    int   in[SGP_MAX_PEERS];
    int   out[SGP_MAX_PEERS];
    float self_w;
    float in_w[SGP_MAX_PEERS];
};

__device__ __forceinline__ void load_row(const SgpArgs& a, uint32_t step_like, RowInfo& r) {
    const uint32_t row = (step_like + a.st->phase_base) % (uint32_t)a.period;
    const int*   t = a.table  + row * SGP_TABLE_ROW;
    const float* w = a.wtable + row * SGP_WTABLE_ROW;
    r.n_in = t[0];
    r.n_out = t[1];
#pragma unroll
    for (int k = 0; k < SGP_MAX_PEERS; ++k) {
        r.in[k]   = t[2 + k];
        r.out[k]  = t[2 + SGP_MAX_PEERS + k];
        r.in_w[k] = w[1 + k];
    }
    r.self_w = w[0];
}

__device__ __forceinline__ float4 fma4(float4 a, float s, float4 b) {
    return make_float4(fmaf(a.x, s, b.x), fmaf(a.y, s, b.y), fmaf(a.z, s, b.z), fmaf(a.w, s, b.w));
}
__device__ __forceinline__ float4 mul4(float4 a, float s) {
    return make_float4(a.x * s, a.y * s, a.z * s, a.w * s);
}

// SGD with momentum on the push-sum numerator (torch.optim.SGD semantics,
// dampening 0): d = g + wd*x ; m = mu*m + d ; x -= lr * (nesterov ? d + mu*m : m)
__device__ __forceinline__ void sgd1(float& x, float g, float& m, float lr, float mu,
                                     float wd, float nesterov) {
    const float d = fmaf(wd, x, g);
    m = fmaf(mu, m, d);
    const float upd = (nesterov != 0.f) ? fmaf(mu, m, d) : m;
    x = fmaf(-lr, upd, x);
}

// Last-CTA bookkeeping shared by the kernels: returns true in thread 0 of the
// CTA that finishes last.
__device__ __forceinline__ bool cta_done_is_last(SgpState* st) {
    __threadfence();
    const uint32_t prev = atomicAdd(&st->done_ctas, 1u);
    if (prev == gridDim.x - 1) {
        __threadfence();
        return true;
    }
    return false;
}

}  // namespace

// ---------------------------------------------------------------------------
// Fused step kernel
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(SGP_THREADS, 2)
sgp_step_kernel(const SgpArgs a)
{
    __shared__ float s_wn;        // new push-sum weight
    __shared__ int   s_ok;

    SgpState* st = a.st;
    const uint32_t step   = *((volatile uint32_t*)&st->step);
    const uint32_t parity = step & 1u;
    // AD-PSGD: the mode bits come from the device-side round state machine (what the preceding
    // sgp_bilat_decide_kernel decided); nothing to do -> the whole grid exits at once
    const bool from_state = (a.flags & SGP_F_FROM_STATE) != 0;
    const uint32_t flags  = from_state
        ? ((a.flags & (SGP_F_SHADOW | SGP_F_GRAD_BF16)) | *((volatile uint32_t*)&st->bilat_cmd))
        : a.flags;
    if (from_state && (flags & (SGP_F_PHASE1 | SGP_F_PHASE2)) == 0u) return;
    const int      tid    = threadIdx.x;
    const int      b      = blockIdx.x;
    const long long nchunks = a.n / SGP_CHUNK;

    RowInfo row;
    load_row(a, step, row);

    const float w0 = *((volatile float*)&st->ps_weight[parity]);
    const float wmul = (flags & SGP_F_IN_NUMER) ? 1.f : w0;   // z -> numerator factor
    const float wres = (flags & SGP_F_FOLD_RES) ? *((volatile float*)&st->res_weight) : 0.f;
    const float rscale = (flags & SGP_F_FOLD_RES) ? *((volatile float*)&st->res_scale) : 1.f;
    const float w1 = w0 + wres;                    // weight of the published numerator

    SgpSignalPad* mypad = a.pads[a.rank];
    float* my_out = a.outboxes ? (a.outboxes[a.rank] + (size_t)parity * a.n) : nullptr;

    const SgpHyper hp = *a.hyper;
    const uint64_t pol_first = l2_evict_first_policy();
    const uint64_t pol_last = l2_evict_last_policy();
    const bool do_sgd = (flags & SGP_F_SGD) && (hp.do_sgd != 0.f);

    // Work decomposition: this CTA owns chunks b, b+G, b+2G, ...; they are cut into
    // K contiguous SEGMENTS.  For each segment the CTA runs phase 1 (local update +
    // publish, HBM-bound), releases a per-CTA progress counter
    //        pub_seq[b] = step * SGP_SEQ_STRIDE + seg + 1
    // and immediately runs phase 2 (pull + mix, NVLink-bound) on the same segment.
    // CTAs sharing an SM drift apart, so one CTA's NVLink phase overlaps another's
    // HBM phase and the kernel approaches max(HBM time, NVLink time) instead of
    // their sum; the own-term re-read of phase 2 always hits L2.
    const long long my_chunks = (nchunks > b) ? (nchunks - 1 - b) / gridDim.x + 1 : 0;
    int K = a.segments < 1 ? 1 : a.segments;
    if (K > SGP_SEQ_STRIDE - 1) K = SGP_SEQ_STRIDE - 1;
    const uint32_t seq_base = step * (uint32_t)SGP_SEQ_STRIDE;

    if ((flags & SGP_F_PHASE1) && (flags & SGP_F_PUBLISH) && step >= st->ack_from + 2u) {
        // WAR fence: outbox[parity] was last read at step-2 by that step's
        // out-neighbours; wait for their acks before overwriting it.
        if (tid == 0) {
            RowInfo prev;
            load_row(a, step - 2u, prev);
            int ok = 1;
            for (int k = 0; k < prev.n_out; ++k) {
                const int o = prev.out[k];
                if (o == a.rank || o < 0) continue;
                ok &= spin_wait_geq(&mypad->ack_seq[o], step - 1u, st, a.timeout_ns,
                                    SGP_ERR_TIMEOUT_ACK) ? 1 : 0;
            }
            s_ok = ok;
        }
        __syncthreads();
    }

    const float inv_w1 = 1.f / w1;
    const bool write_z = !(flags & SGP_F_PHASE2) && !(flags & SGP_F_KEEP_Z);
    // overlap publish keeps the self-loop share locally (w <- self_w * w1); a
    // snapshot-only publish (AD-PSGD) leaves the weight alone
    float w_next = ((flags & SGP_F_PUBLISH) && !(flags & SGP_F_KEEP_Z)) ? row.self_w * w1 : w1;
    float inv_wn = 1.f;
    bool pull_ok = true;
    const float* peer_out[SGP_MAX_PEERS];
#pragma unroll
    for (int k = 0; k < SGP_MAX_PEERS; ++k)
        peer_out[k] = ((flags & SGP_F_PHASE2) && k < row.n_in && row.in[k] >= 0)
                          ? a.outboxes[row.in[k]] + (size_t)parity * a.n : nullptr;

    for (int seg = 0; seg < K; ++seg) {
        const long long it_lo = my_chunks * seg / K;
        const long long it_hi = my_chunks * (seg + 1) / K;

        // ---------------- phase 1: local update + publish ------------------
        if (flags & SGP_F_PHASE1) {
            for (long long it = it_lo; it < it_hi; ++it) {
                const long long c = b + it * gridDim.x;
                const long long base = c * SGP_CHUNK + (long long)tid * SGP_VEC;
                float4 x[SGP_UNROLL], g[SGP_UNROLL], m[SGP_UNROLL], r[SGP_UNROLL];
#pragma unroll
                for (int u = 0; u < SGP_UNROLL; ++u) {
                    const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                    x[u] = ld_once_f4(reinterpret_cast<const float4*>(a.z + i), pol_first);
                    if (do_sgd) {
                        if (flags & SGP_F_GRAD_BF16)
                            g[u] = bf16x4_to_f4(ld_once_u2(reinterpret_cast<const uint2*>(
                                       reinterpret_cast<const __nv_bfloat16*>(a.g) + i), pol_first));
                        else
                            g[u] = ld_once_f4(reinterpret_cast<const float4*>(
                                       reinterpret_cast<const float*>(a.g) + i), pol_first);
                        if (a.g2 != nullptr) {
                            const float4 h = ld_once_f4(reinterpret_cast<const float4*>(a.g2 + i), pol_first);
                            g[u].x += h.x; g[u].y += h.y; g[u].z += h.z; g[u].w += h.w;
                        }
                        m[u] = ld_once_f4(reinterpret_cast<const float4*>(a.m + i), pol_first);
                    }
                    if (flags & SGP_F_FOLD_RES)
                        r[u] = ld_once_f4(reinterpret_cast<const float4*>(a.residual + i), pol_first);
                }
#pragma unroll
                for (int u = 0; u < SGP_UNROLL; ++u) {
                    const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                    float4 xv = mul4(x[u], wmul);               // numerator (exact if w == 1)
                    if (do_sgd) {
                        float4 gv = mul4(g[u], hp.grad_scale);
                        float4 mv = m[u];
                        sgd1(xv.x, gv.x, mv.x, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                        sgd1(xv.y, gv.y, mv.y, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                        sgd1(xv.z, gv.z, mv.z, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                        sgd1(xv.w, gv.w, mv.w, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                        st_f4(reinterpret_cast<float4*>(a.m + i), mv);
                        if (flags & SGP_F_ZERO_GRAD) {
                            if (flags & SGP_F_GRAD_BF16)
                                st_u2(reinterpret_cast<uint2*>(
                                          reinterpret_cast<__nv_bfloat16*>(a.g) + i), make_uint2(0u, 0u));
                            else
                                st_f4(reinterpret_cast<float4*>(reinterpret_cast<float*>(a.g) + i),
                                      make_float4(0.f, 0.f, 0.f, 0.f));
                            if (a.g2 != nullptr)
                                st_f4(reinterpret_cast<float4*>(a.g2 + i), make_float4(0.f, 0.f, 0.f, 0.f));
                        }
                    }
                    if (flags & SGP_F_FOLD_RES) {      // (rscale: 1 after a gather kernel, the edge weight after a DMA gather)
                        xv.x = fmaf(r[u].x, rscale, xv.x); xv.y = fmaf(r[u].y, rscale, xv.y);
                        xv.z = fmaf(r[u].z, rscale, xv.z); xv.w = fmaf(r[u].w, rscale, xv.w);
                    }
                    if (flags & SGP_F_PUBLISH)   // keep the outbox in L2 for phase 2 / peers
                        st_hint_f4(reinterpret_cast<float4*>(my_out + i), xv, pol_last);
                    if (write_z) {
                        const float4 zv = mul4(xv, inv_w1);
                        st_f4(reinterpret_cast<float4*>(a.z + i), zv);
                        if (flags & SGP_F_SHADOW)
                            st_u2(reinterpret_cast<uint2*>(a.shadow + i), f4_to_bf16x4(zv));
                    }
                }
            }
            if (flags & SGP_F_PUBLISH) {
                __syncthreads();
                if (tid == 0) {
                    if (seg == 0) st_relaxed_sys_f32(&mypad->psw[parity], w1);  // same value from every CTA
                    __threadfence_system();
                    st_release_sys(&mypad->pub_seq[b], seq_base + (uint32_t)seg + 1u);
                }
            }
        }

        // ---------------- phase 2: pull + mix ------------------------------
        if (flags & SGP_F_PHASE2) {
            if (tid == 0) {
                int ok = 1;
                float wn = row.self_w * w1;
                for (int k = 0; k < row.n_in; ++k) {
                    const int j = row.in[k];
                    if (j < 0) continue;
                    const SgpSignalPad* pj = a.pads[j];
                    ok &= spin_wait_geq(&pj->pub_seq[b], seq_base + (uint32_t)seg + 1u, st,
                                        a.timeout_ns, SGP_ERR_TIMEOUT_PUB) ? 1 : 0;
                    if (seg == 0) wn = fmaf(row.in_w[k], ld_relaxed_sys_f32(&pj->psw[parity]), wn);
                }
                if (seg == 0) s_wn = wn;
                s_ok = ok;
            }
            __syncthreads();
            if (seg == 0) {
                w_next = s_wn;
                inv_wn = 1.f / s_wn;
            }
            pull_ok = pull_ok && (s_ok != 0);
            if (pull_ok) {
                for (long long it = it_lo; it < it_hi; ++it) {
                    const long long c = b + it * gridDim.x;
                    const long long base = c * SGP_CHUNK + (long long)tid * SGP_VEC;
                    float4 acc[SGP_UNROLL];
                    float4 pv[SGP_UNROLL];
#pragma unroll
                    for (int u = 0; u < SGP_UNROLL; ++u) {
                        const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                        // own term: the snapshot this CTA just published (L2-resident),
                        // or (AD-PSGD) the live parameters, which may already carry
                        // newer local SGD updates
                        const float* own = (flags & SGP_F_SELF_FROM_Z) ? a.z : my_out;
                        acc[u] = mul4(ld_once_f4(reinterpret_cast<const float4*>(own + i), pol_first),
                                      (flags & SGP_F_SELF_FROM_Z) ? row.self_w * w0 : row.self_w);
                    }
                    // peer loads: all UNROLL requests of one peer in flight together
                    for (int k = 0; k < row.n_in; ++k) {
                        const float* po = peer_out[k];
                        if (po == nullptr) continue;
#pragma unroll
                        for (int u = 0; u < SGP_UNROLL; ++u) {
                            const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                            pv[u] = ld_stream_f4(reinterpret_cast<const float4*>(po + i));
                        }
                        const float wk = row.in_w[k];
#pragma unroll
                        for (int u = 0; u < SGP_UNROLL; ++u) acc[u] = fma4(pv[u], wk, acc[u]);
                    }
#pragma unroll
                    for (int u = 0; u < SGP_UNROLL; ++u) {
                        const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                        const float4 zv = mul4(acc[u], inv_wn);
                        st_f4(reinterpret_cast<float4*>(a.z + i), zv);
                        if (flags & SGP_F_SHADOW)
                            st_u2(reinterpret_cast<uint2*>(a.shadow + i), f4_to_bf16x4(zv));
                    }
                }
            }
            else if (!(flags & SGP_F_SELF_FROM_Z) && (flags & SGP_F_PHASE1)) {
                // an in-neighbour timed out: "every in-message of this round was lost" -- de-bias the
                // numerator this CTA published (a valid push-sum state) instead of leaving the
                // pre-SGD parameters behind; the sticky status word makes the host raise
                const float inv_own = 1.f / w1;
                for (long long it = it_lo; it < it_hi; ++it) {
                    const long long c = b + it * gridDim.x;
                    const long long base = c * SGP_CHUNK + (long long)tid * SGP_VEC;
#pragma unroll
                    for (int u = 0; u < SGP_UNROLL; ++u) {
                        const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                        const float4 zv = mul4(ld_once_f4(reinterpret_cast<const float4*>(my_out + i), pol_first),
                                               inv_own);
                        st_f4(reinterpret_cast<float4*>(a.z + i), zv);
                        if (flags & SGP_F_SHADOW)
                            st_u2(reinterpret_cast<uint2*>(a.shadow + i), f4_to_bf16x4(zv));
                    }
                }
            }
            __syncthreads();     // s_ok / s_wn are rewritten by the next segment
        }
    }

    // ---------------- epilogue: last CTA publishes state + acks ------------
    __syncthreads();
    if (tid == 0 && cta_done_is_last(st)) {
        if (flags & SGP_F_PHASE2) {
            for (int k = 0; k < row.n_in; ++k) {
                const int j = row.in[k];
                if (j < 0 || j == a.rank) continue;
                st_release_sys(&a.pads[j]->ack_seq[a.rank], step + 1u);
            }
        }
        const bool rotate = !(flags & SGP_F_NO_ROTATE);
        *((volatile float*)&st->ps_weight[rotate ? (parity ^ 1u) : parity]) = w_next;
        if (flags & SGP_F_FOLD_RES) *((volatile float*)&st->res_weight) = 0.f;
        *((volatile uint32_t*)&st->done_ctas) = 0u;
        if (rotate) *((volatile uint32_t*)&st->step) = step + 1u;
        if (from_state) {                       // bilateral round bookkeeping
            if (rotate) {                       // round complete
                st->bilat_published = 0u;
                st->bilat_round += 1u;
            } else if (flags & SGP_F_PUBLISH) {
                st->bilat_published = 1u;       // snapshot is out; the pull follows in a later launch
            }
            st->bilat_cmd = 0u;
        }
        __threadfence();
    }
}

// ---------------------------------------------------------------------------
// Overlap-SGP gather: residual = sum_k in_w[k] * outbox_k[parity]   (side stream)
// Runs after the local publish kernel of the same step, i.e. st->step == s+1.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(SGP_THREADS, 2)
sgp_gather_kernel(const SgpArgs a, const int pub_grid)
{
    __shared__ int s_ok;
    SgpState* st = a.st;
    const uint32_t s      = *((volatile uint32_t*)&st->step) - 1u;
    const uint32_t parity = s & 1u;
    const int tid = threadIdx.x;
    const long long nchunks = a.n / SGP_CHUNK;

    RowInfo row;
    load_row(a, s, row);
    int segs = a.segments < 1 ? 1 : a.segments;
    if (segs > SGP_SEQ_STRIDE - 1) segs = SGP_SEQ_STRIDE - 1;

    // every CTA waits for ALL publisher CTAs of every in-neighbour (block-parallel poll)
    if (tid == 0) s_ok = 1;
    __syncthreads();
    for (int k = 0; k < row.n_in; ++k) {
        const int j = row.in[k];
        if (j < 0) continue;
        const SgpSignalPad* pj = a.pads[j];
        for (int f = tid; f < pub_grid; f += SGP_THREADS)
            if (!spin_wait_geq(&pj->pub_seq[f], s * (uint32_t)SGP_SEQ_STRIDE + (uint32_t)segs, st,
                               a.timeout_ns, SGP_ERR_TIMEOUT_PUB))
                s_ok = 0;
    }
    __syncthreads();

    if (s_ok) {
        const float* peer_out[SGP_MAX_PEERS];
#pragma unroll
        for (int k = 0; k < SGP_MAX_PEERS; ++k)
            peer_out[k] = (k < row.n_in && row.in[k] >= 0)
                              ? a.outboxes[row.in[k]] + (size_t)parity * a.n : nullptr;
        for (long long c = blockIdx.x; c < nchunks; c += gridDim.x) {
            const long long base = c * SGP_CHUNK + (long long)tid * SGP_VEC;
            float4 acc[SGP_UNROLL], pv[SGP_UNROLL];
#pragma unroll
            for (int u = 0; u < SGP_UNROLL; ++u) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int k = 0; k < row.n_in; ++k) {
                const float* po = peer_out[k];
                if (po == nullptr) continue;
#pragma unroll
                for (int u = 0; u < SGP_UNROLL; ++u)
                    pv[u] = ld_stream_f4(reinterpret_cast<const float4*>(
                                po + base + (long long)u * SGP_THREADS * SGP_VEC));
#pragma unroll
                for (int u = 0; u < SGP_UNROLL; ++u) acc[u] = fma4(pv[u], row.in_w[k], acc[u]);
            }
#pragma unroll
            for (int u = 0; u < SGP_UNROLL; ++u)
                st_f4(reinterpret_cast<float4*>(a.residual + base +
                                                (long long)u * SGP_THREADS * SGP_VEC), acc[u]);
        }
    }

    __syncthreads();
    if (tid == 0 && cta_done_is_last(st)) {
        float wr = 0.f;
        for (int k = 0; k < row.n_in; ++k) {
            const int j = row.in[k];
            if (j < 0) continue;
            wr = fmaf(row.in_w[k], ld_relaxed_sys_f32(&a.pads[j]->psw[parity]), wr);
            if (j != a.rank) st_release_sys(&a.pads[j]->ack_seq[a.rank], s + 1u);
        }
        *((volatile float*)&st->res_weight) = s_ok ? wr : 0.f;
        *((volatile float*)&st->res_scale) = 1.f;
        *((volatile uint32_t*)&st->done_ctas) = 0u;
        __threadfence();
    }
}

// ---------------------------------------------------------------------------
// Overlap-SGP gather, TMA variant.  The gather runs on a side stream next to the
// forward/backward pass, so it should saturate NVLink from as FEW SMs as possible.
// Register-staged loads need ~300 CTAs of in-flight 16-byte requests to cover the
// ~2 us NVLink latency; here one elected thread per CTA keeps a ring of
// SGP_TMA_STAGES x 16 KB bulk copies (cp.async.bulk, global[peer] -> shared,
// mbarrier complete_tx) in flight, i.e. ~100 KB per CTA instead of ~16 KB, and the
// whole CTA only touches the data once it has landed in shared memory.
// ---------------------------------------------------------------------------
#define SGP_TMA_STAGES 6
#define SGP_TMA_BYTES  (SGP_CHUNK * 4)      // one 4096-float chunk = 16 KB per stage

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(SGP_THREADS, 1)
sgp_gather_tma_kernel(const SgpArgs a, const int pub_grid)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* ring = reinterpret_cast<float*>(smem_raw);                       // [STAGES][CHUNK]
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + SGP_TMA_STAGES * SGP_TMA_BYTES);
    __shared__ int s_ok;

    SgpState* st = a.st;
    const uint32_t s      = *((volatile uint32_t*)&st->step) - 1u;
    const uint32_t parity = s & 1u;
    const int tid = threadIdx.x;
    const long long nchunks = a.n / SGP_CHUNK;

    RowInfo row;
    load_row(a, s, row);
    int segs = a.segments < 1 ? 1 : a.segments;
    if (segs > SGP_SEQ_STRIDE - 1) segs = SGP_SEQ_STRIDE - 1;

    if (tid == 0) {
        s_ok = 1;
        for (int i = 0; i < SGP_TMA_STAGES; ++i) mbar_init(&full[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    for (int k = 0; k < row.n_in; ++k) {
        const int j = row.in[k];
        if (j < 0) continue;
        const SgpSignalPad* pj = a.pads[j];
        for (int f = tid; f < pub_grid; f += SGP_THREADS)
            if (!spin_wait_geq(&pj->pub_seq[f], s * (uint32_t)SGP_SEQ_STRIDE + (uint32_t)segs, st,
                               a.timeout_ns, SGP_ERR_TIMEOUT_PUB))
                s_ok = 0;
    }
    __syncthreads();

    const int n_in = row.n_in;
    const long long my_chunks = (nchunks > blockIdx.x) ? (nchunks - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    const long long items = s_ok ? my_chunks * n_in : 0;     // (chunk, in-peer) pairs, peer fastest

    auto issue = [&](long long item) {
        const long long it = item / n_in;
        const int k = (int)(item - it * n_in);
        const long long c = blockIdx.x + it * gridDim.x;
        const int stage = (int)(item % SGP_TMA_STAGES);
        const float* src = a.outboxes[row.in[k]] + (size_t)parity * a.n + c * SGP_CHUNK;
        mbar_expect_tx(&full[stage], SGP_TMA_BYTES);
        tma_load_1d(ring + (size_t)stage * SGP_CHUNK, src, SGP_TMA_BYTES, &full[stage]);
    };

    if (tid == 0)
        for (long long i = 0; i < items && i < SGP_TMA_STAGES; ++i) issue(i);

    float4 acc[SGP_UNROLL];
    for (long long item = 0; item < items; ++item) {
        const long long it = item / n_in;
        const int k = (int)(item - it * n_in);
        const int stage = (int)(item % SGP_TMA_STAGES);
        mbar_wait(&full[stage], (uint32_t)((item / SGP_TMA_STAGES) & 1));
        const float4* src = reinterpret_cast<const float4*>(ring + (size_t)stage * SGP_CHUNK);
        const float wk = row.in_w[k];
#pragma unroll
        for (int u = 0; u < SGP_UNROLL; ++u) {
            const float4 v = src[tid + u * SGP_THREADS];
            acc[u] = (k == 0) ? mul4(v, wk) : fma4(v, wk, acc[u]);
        }
        if (k == n_in - 1) {
            const long long c = blockIdx.x + it * gridDim.x;
            float4* dst = reinterpret_cast<float4*>(a.residual + c * SGP_CHUNK);
#pragma unroll
            for (int u = 0; u < SGP_UNROLL; ++u) st_f4(dst + tid + u * SGP_THREADS, acc[u]);
        }
        __syncthreads();                         // every thread is done with this stage
        if (tid == 0 && item + SGP_TMA_STAGES < items) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic reads -> async write
            issue(item + SGP_TMA_STAGES);
        }
    }

    __syncthreads();
    if (tid == 0 && cta_done_is_last(st)) {
        float wr = 0.f;
        for (int k = 0; k < row.n_in; ++k) {
            const int j = row.in[k];
            if (j < 0) continue;
            wr = fmaf(row.in_w[k], ld_relaxed_sys_f32(&a.pads[j]->psw[parity]), wr);
            if (j != a.rank) st_release_sys(&a.pads[j]->ack_seq[a.rank], s + 1u);
        }
        *((volatile float*)&st->res_weight) = s_ok ? wr : 0.f;
        *((volatile float*)&st->res_scale) = 1.f;
        *((volatile uint32_t*)&st->done_ctas) = 0u;
        __threadfence();
    }
}

// ---------------------------------------------------------------------------
// Fused step kernel, warp-specialised + TMA-fed variant (the SGP / D-PSGD hot path).
//
// sgp_step_kernel pulls the peers' outboxes with register-staged 16-byte loads: every
// consumer thread has 4 x 16 B in flight and the CTA alternates between an HBM-bound phase 1
// and an NVLink-bound phase 2 (0.257 ms at ResNet-50 size on 2 GPUs = 52 % of the NVLink
// roofline, profiles/README.md).  Here the two phases run on different warps of the same CTA:
//
//   warps 0-7 (consumers)  for seg = 0..K:   phase 1 of segment `seg`   (SGD + publish, HBM)
//                                            phase 2 of segment `seg-1` (mix + de-bias)
//                          phase 2 reads the peers' data from SHARED MEMORY, where it has
//                          been landing while phase 1 of the next segment was streaming HBM
//   warp 8 lane 0 (producer) per segment: acquire the in-neighbours' publish flags, then keep
//                          a ring of PIPE_STAGES x 16 KB bulk copies (cp.async.bulk,
//                          peer global -> shared, mbarrier complete_tx) in flight over NVLink
//
// so the NVLink stream starts as soon as the first segment of the peer is published and
// never waits for a consumer register to free up; the consumers never wait for NVLink
// latency.  Flags, outbox layout, acks and the last-CTA epilogue are those of
// sgp_step_kernel (gather / probe / the old kernel interoperate with it); the grid must be
// the same on all ranks (flags are matched by CTA index).
//
// (Tried and rejected, round 2: splitting the consumers into a phase-1 group and a phase-2 group of
// four warps each so that both streams run concurrently inside a CTA -- 0.298 ms vs 0.254 ms for
// this version on 2 GPUs: four warps per stream no longer cover the HBM / shared-memory latencies.)
//
// A timed-out flag wait does not leave stale parameters behind: the producer marks the CTA
// failed, completes its barriers without data, and the consumers de-bias their own published
// numerator instead (z = x_own / w1, i.e. "every in-message of this round was lost" -- a valid
// push-sum state); the sticky status word makes the host raise at its next poll.
// ---------------------------------------------------------------------------
#define PIPE_STAGES    4
#define PIPE_CONSUMERS SGP_THREADS                 // 256: the chunk decomposition of sgp_step_kernel
#define PIPE_THREADS   (PIPE_CONSUMERS + 32)
#define PIPE_SMEM      (PIPE_STAGES * SGP_TMA_BYTES + 2 * PIPE_STAGES * 8 + 64)

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}

// 9 warps x 2 CTAs per SM: the register file is split over 4 sub-partitions (16 K registers
// each), so 18 warps only fit at <= 102 registers per thread -- __launch_bounds__(288, 2) makes
// ptxas pick 96.  (At 112 registers ncu showed launch__occupancy_limit_registers = 1 block and
// the kernel ran one CTA per SM, profiles/step_pipe_2gpu_nvlink_ncu_r2_v1.csv.)
__global__ void __launch_bounds__(PIPE_THREADS, 2)
sgp_step_pipe_kernel(const SgpArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* ring = reinterpret_cast<float*>(smem_raw);                          // [STAGES][CHUNK]
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + PIPE_STAGES * SGP_TMA_BYTES);
    uint64_t* empty = full + PIPE_STAGES;
    uint64_t* wbar = empty + PIPE_STAGES;            // new push-sum weight is known
    __shared__ float s_wn;
    __shared__ int   s_ok;                            // WAR fence outcome (consumers)
    __shared__ volatile int s_fail;                   // producer: an in-neighbour timed out

    SgpState* st = a.st;
    const uint32_t step   = *((volatile uint32_t*)&st->step);
    const uint32_t parity = step & 1u;
    const uint32_t flags  = a.flags;
    const int      tid    = threadIdx.x;
    const int      warp   = tid >> 5;
    const int      b      = blockIdx.x;
    const long long nchunks = a.n / SGP_CHUNK;

    RowInfo row;
    load_row(a, step, row);

    const float w0 = *((volatile float*)&st->ps_weight[parity]);
    const float wmul = (flags & SGP_F_IN_NUMER) ? 1.f : w0;
    const float w1 = w0;                              // (no residual fold in the synchronous step)

    SgpSignalPad* mypad = a.pads[a.rank];
    float* my_out = a.outboxes[a.rank] + (size_t)parity * a.n;

    const long long my_chunks = (nchunks > b) ? (nchunks - 1 - b) / gridDim.x + 1 : 0;
    int K = a.segments < 1 ? 1 : a.segments;
    if (K > SGP_SEQ_STRIDE - 1) K = SGP_SEQ_STRIDE - 1;
    const uint32_t seq_base = step * (uint32_t)SGP_SEQ_STRIDE;

    // compacted in-neighbour list (table entries < 0 are holes)
    int n_in = 0;
    int in_rank[SGP_MAX_PEERS];
    float in_w[SGP_MAX_PEERS];
#pragma unroll
    for (int k = 0; k < SGP_MAX_PEERS; ++k)
        if (k < row.n_in && row.in[k] >= 0) { in_rank[n_in] = row.in[k]; in_w[n_in] = row.in_w[k]; ++n_in; }

    if (tid == 0) {
        for (int i = 0; i < PIPE_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], PIPE_CONSUMERS / 32); }
        mbar_init(wbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        s_fail = 0;
        s_ok = 1;
    }
    __syncthreads();

    if (warp == PIPE_CONSUMERS / 32) {
        // ============================ producer ============================
        if ((tid & 31) == 0) {
            int stage = 0;
            uint32_t phase = 0;
            bool ok = true;
            float wn = row.self_w * w1;
            for (int seg = 0; seg < K; ++seg) {
                for (int k = 0; k < n_in && ok; ++k) {
                    const SgpSignalPad* pj = a.pads[in_rank[k]];
                    ok = spin_wait_geq(&pj->pub_seq[b], seq_base + (uint32_t)seg + 1u, st, a.timeout_ns,
                                       SGP_ERR_TIMEOUT_PUB);
                    if (ok && seg == 0) wn = fmaf(in_w[k], ld_relaxed_sys_f32(&pj->psw[parity]), wn);
                }
                if (!ok) s_fail = 1;
                if (seg == 0) {
                    s_wn = ok ? wn : row.self_w * w1;
                    __threadfence_block();
                    mbar_arrive(wbar);
                }
                const long long it_lo = my_chunks * seg / K, it_hi = my_chunks * (seg + 1) / K;
                for (long long it = it_lo; it < it_hi; ++it) {
                    const long long c = b + it * gridDim.x;
                    for (int k = 0; k < n_in; ++k) {
                        mbar_wait(&empty[stage], phase ^ 1u);
                        if (ok) {
                            const float* src = a.outboxes[in_rank[k]] + (size_t)parity * a.n + c * SGP_CHUNK;
                            mbar_expect_tx(&full[stage], SGP_TMA_BYTES);
                            tma_load_1d(ring + (size_t)stage * SGP_CHUNK, src, SGP_TMA_BYTES, &full[stage]);
                        } else {
                            mbar_arrive(&full[stage]);           // nothing will land: release the consumers
                        }
                        if (++stage == PIPE_STAGES) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
        __syncwarp();
    } else {
        // ============================ consumers ============================
        const SgpHyper hp = *a.hyper;
        const uint64_t pol_first = l2_evict_first_policy();
        const uint64_t pol_last = l2_evict_last_policy();
        const bool do_sgd = (flags & SGP_F_SGD) && (hp.do_sgd != 0.f);
        const int lane = tid & 31;

        if (step >= st->ack_from + 2u) {
            // WAR fence: outbox[parity] was last read at step-2 by that step's out-neighbours
            if (tid == 0) {
                RowInfo prev;
                load_row(a, step - 2u, prev);
                int ok = 1;
                for (int k = 0; k < prev.n_out; ++k) {
                    const int o = prev.out[k];
                    if (o == a.rank || o < 0) continue;
                    ok &= spin_wait_geq(&mypad->ack_seq[o], step - 1u, st, a.timeout_ns, SGP_ERR_TIMEOUT_ACK) ? 1 : 0;
                }
                s_ok = ok;
            }
            asm volatile("bar.sync 1, %0;" :: "n"(PIPE_CONSUMERS) : "memory");
        }

        int cstage = 0;
        uint32_t cphase = 0;
        float inv_wn = 1.f;
        const float inv_w1 = 1.f / w1;

        for (int seg = 0; seg <= K; ++seg) {
            // ---------------- phase 1 of segment `seg`: local update + publish ----------------
            if (seg < K) {
                const long long it_lo = my_chunks * seg / K, it_hi = my_chunks * (seg + 1) / K;
                for (long long it = it_lo; it < it_hi; ++it) {
                    const long long c = b + it * gridDim.x;
                    const long long base = c * SGP_CHUNK + (long long)tid * SGP_VEC;
                    float4 x[SGP_UNROLL], g[SGP_UNROLL], m[SGP_UNROLL];
#pragma unroll
                    for (int u = 0; u < SGP_UNROLL; ++u) {
                        const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                        x[u] = ld_once_f4(reinterpret_cast<const float4*>(a.z + i), pol_first);
                        if (do_sgd) {
                            if (flags & SGP_F_GRAD_BF16)
                                g[u] = bf16x4_to_f4(ld_once_u2(reinterpret_cast<const uint2*>(
                                           reinterpret_cast<const __nv_bfloat16*>(a.g) + i), pol_first));
                            else
                                g[u] = ld_once_f4(reinterpret_cast<const float4*>(
                                           reinterpret_cast<const float*>(a.g) + i), pol_first);
                            if (a.g2 != nullptr) {
                                const float4 h = ld_once_f4(reinterpret_cast<const float4*>(a.g2 + i), pol_first);
                                g[u].x += h.x; g[u].y += h.y; g[u].z += h.z; g[u].w += h.w;
                            }
                            m[u] = ld_once_f4(reinterpret_cast<const float4*>(a.m + i), pol_first);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < SGP_UNROLL; ++u) {
                        const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                        float4 xv = mul4(x[u], wmul);
                        if (do_sgd) {
                            float4 gv = mul4(g[u], hp.grad_scale);
                            float4 mv = m[u];
                            sgd1(xv.x, gv.x, mv.x, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                            sgd1(xv.y, gv.y, mv.y, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                            sgd1(xv.z, gv.z, mv.z, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                            sgd1(xv.w, gv.w, mv.w, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                            st_f4(reinterpret_cast<float4*>(a.m + i), mv);
                            if (flags & SGP_F_ZERO_GRAD) {
                                if (flags & SGP_F_GRAD_BF16)
                                    st_u2(reinterpret_cast<uint2*>(
                                              reinterpret_cast<__nv_bfloat16*>(a.g) + i), make_uint2(0u, 0u));
                                else
                                    st_f4(reinterpret_cast<float4*>(reinterpret_cast<float*>(a.g) + i),
                                          make_float4(0.f, 0.f, 0.f, 0.f));
                                if (a.g2 != nullptr)
                                    st_f4(reinterpret_cast<float4*>(a.g2 + i), make_float4(0.f, 0.f, 0.f, 0.f));
                            }
                        }
                        st_hint_f4(reinterpret_cast<float4*>(my_out + i), xv, pol_last);
                    }
                }
                asm volatile("bar.sync 1, %0;" :: "n"(PIPE_CONSUMERS) : "memory");
                if (tid == 0) {
                    if (seg == 0) st_relaxed_sys_f32(&mypad->psw[parity], w1);
                    __threadfence_system();
                    st_release_sys(&mypad->pub_seq[b], seq_base + (uint32_t)seg + 1u);
                }
            }
            // ---------------- phase 2 of segment `seg - 1`: mix + de-bias ----------------
            if (seg >= 1) {
                const int ps = seg - 1;
                if (ps == 0) {
                    mbar_wait(wbar, 0);
                    inv_wn = 1.f / s_wn;
                }
                const long long it_lo = my_chunks * ps / K, it_hi = my_chunks * (ps + 1) / K;
                for (long long it = it_lo; it < it_hi; ++it) {
                    const long long c = b + it * gridDim.x;
                    const long long base = c * SGP_CHUNK + (long long)tid * SGP_VEC;
                    float4 acc[SGP_UNROLL];
#pragma unroll
                    for (int u = 0; u < SGP_UNROLL; ++u) {
                        const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                        acc[u] = mul4(ld_once_f4(reinterpret_cast<const float4*>(my_out + i), pol_first),   // L2 hit
                                      row.self_w);
                    }
                    for (int k = 0; k < n_in; ++k) {
                        mbar_wait(&full[cstage], cphase);
                        const float4* src = reinterpret_cast<const float4*>(ring + (size_t)cstage * SGP_CHUNK);
                        const float wk = in_w[k];
#pragma unroll
                        for (int u = 0; u < SGP_UNROLL; ++u) acc[u] = fma4(src[tid + u * SGP_THREADS], wk, acc[u]);
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&empty[cstage]);     // this warp is done with the stage
                        if (++cstage == PIPE_STAGES) { cstage = 0; cphase ^= 1u; }
                    }
                    const bool failed = s_fail != 0;           // (rare: re-read the own numerator)
#pragma unroll
                    for (int u = 0; u < SGP_UNROLL; ++u) {
                        const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                        const float4 zv = failed
                            ? mul4(ld_once_f4(reinterpret_cast<const float4*>(my_out + i), pol_first), inv_w1)
                            : mul4(acc[u], inv_wn);
                        st_f4(reinterpret_cast<float4*>(a.z + i), zv);
                        if (flags & SGP_F_SHADOW)
                            st_u2(reinterpret_cast<uint2*>(a.shadow + i), f4_to_bf16x4(zv));
                    }
                }
            }
        }
    }

    // ---------------- epilogue: last CTA publishes state + acks ------------
    __syncthreads();
    if (tid == 0 && cta_done_is_last(st)) {
        for (int k = 0; k < n_in; ++k)
            if (in_rank[k] != a.rank) st_release_sys(&a.pads[in_rank[k]]->ack_seq[a.rank], step + 1u);
        *((volatile float*)&st->ps_weight[parity ^ 1u]) = s_wn;
        *((volatile uint32_t*)&st->done_ctas) = 0u;
        *((volatile uint32_t*)&st->step) = step + 1u;
        __threadfence();
    }
}

// ---------------------------------------------------------------------------
// AD-PSGD passive poll: did the in-neighbour of the current round publish?
// ---------------------------------------------------------------------------
__global__ void sgp_probe_kernel(const SgpArgs a, const int pub_grid, uint32_t* host_flag)
{
    __shared__ int s_all;
    SgpState* st = a.st;
    const uint32_t step = *((volatile uint32_t*)&st->step);
    RowInfo row;
    load_row(a, step, row);
    int segs = a.segments < 1 ? 1 : a.segments;
    if (segs > SGP_SEQ_STRIDE - 1) segs = SGP_SEQ_STRIDE - 1;
    if (threadIdx.x == 0) s_all = 1;
    __syncthreads();
    for (int k = 0; k < row.n_in; ++k) {
        const int j = row.in[k];
        if (j < 0) continue;
        for (int f = threadIdx.x; f < pub_grid; f += blockDim.x)
            if ((int32_t)(ld_acquire_sys(&a.pads[j]->pub_seq[f]) -
                          (step * (uint32_t)SGP_SEQ_STRIDE + (uint32_t)segs)) < 0) s_all = 0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // may outbox[step&1] be overwritten?  (the publish kernel would otherwise
        // spin on these acks; the host checks first so no kernel ever waits)
        uint32_t acks_ok = 1u;
        if (step >= st->ack_from + 2u) {
            RowInfo prev;
            load_row(a, step - 2u, prev);
            for (int k = 0; k < prev.n_out; ++k) {
                const int o = prev.out[k];
                if (o < 0 || o == a.rank) continue;
                if ((int32_t)(ld_acquire_sys(&a.pads[a.rank]->ack_seq[o]) - (step - 1u)) < 0)
                    acks_ok = 0u;
            }
        }
        st->bilat_done = (uint32_t)s_all;
        if (host_flag) {
            ((volatile uint32_t*)host_flag)[0] = (uint32_t)s_all;
            ((volatile uint32_t*)host_flag)[1] = acks_ok;
        }
        __threadfence_system();
    }
}

// ---------------------------------------------------------------------------
// Overlap-SGP gather on the COPY ENGINES (one in-neighbour per step).  A gather kernel on the side
// stream -- even the 32-CTA TMA one -- holds SMs while the forward pass starts: persistent
// one-CTA-per-SM kernels (the tcgen05 GEMMs) and 2-CTA/SM tile loops then wait for "their" SM, and
// the overlap costs more than it hides (bench: OSGP +0.41 ms vs SGP +0.22 ms per step at 2 GPUs,
// profiles/bench_r2_n2_*).  With a single in-neighbour the residual is just a copy of the peer's
// outbox, so:
//     sgp_gather_wait_kernel   ONE CTA: wait for the in-neighbour's publish flags of this step
//     cudaMemcpyAsync          peer outbox -> residual, 100 MB over NVLink on a DMA engine: zero SMs
//     sgp_gather_ack_kernel    ONE thread: residual weight / scale (= the edge weight; applied when
//                              the next publish folds the residual), ack the outbox to its owner
// ---------------------------------------------------------------------------
__global__ void sgp_gather_wait_kernel(const SgpArgs a, const int pub_grid)
{
    SgpState* st = a.st;
    const uint32_t s = *((volatile uint32_t*)&st->step) - 1u;
    RowInfo row;
    load_row(a, s, row);
    int segs = a.segments < 1 ? 1 : a.segments;
    if (segs > SGP_SEQ_STRIDE - 1) segs = SGP_SEQ_STRIDE - 1;
    for (int k = 0; k < row.n_in; ++k) {
        const int j = row.in[k];
        if (j < 0) continue;
        for (int f = threadIdx.x; f < pub_grid; f += blockDim.x)
            spin_wait_geq(&a.pads[j]->pub_seq[f], s * (uint32_t)SGP_SEQ_STRIDE + (uint32_t)segs, st,
                          a.timeout_ns, SGP_ERR_TIMEOUT_PUB);
    }
}

__global__ void sgp_gather_ack_kernel(const SgpArgs a)
{
    SgpState* st = a.st;
    const uint32_t s = *((volatile uint32_t*)&st->step) - 1u;
    const uint32_t parity = s & 1u;
    RowInfo row;
    load_row(a, s, row);
    const bool ok = *((volatile uint32_t*)&st->status) == SGP_OK;
    float wr = 0.f, scale = 0.f;
    __threadfence_system();                         // the DMA copy before this kernel has completed
    for (int k = 0; k < row.n_in; ++k) {
        const int j = row.in[k];
        if (j < 0) continue;
        scale = row.in_w[k];                        // (single in-neighbour: enforced by the host)
        wr = fmaf(row.in_w[k], ld_relaxed_sys_f32(&a.pads[j]->psw[parity]), wr);
        if (j != a.rank) st_release_sys(&a.pads[j]->ack_seq[a.rank], s + 1u);
    }
    *((volatile float*)&st->res_weight) = ok ? wr : 0.f;
    *((volatile float*)&st->res_scale) = ok ? scale : 0.f;
    __threadfence();
}

// ---------------------------------------------------------------------------
// AD-PSGD round state machine, device side.  One CTA decides what the NEXT worker launch
// (sgp_step_kernel with SGP_F_FROM_STATE) does, from flags only:
//   * active ranks publish their snapshot unconditionally, passive ranks only once their
//     partner's snapshot of this round is visible (gossip/gossiper.py:290-316);
//   * nobody publishes before the readers of round r-2 released the outbox half;
//   * the pull (x <- 1/2 (x_now + x_partner), ack, advance) runs once both snapshots are out;
//   * waiting for the partner is BOUNDED (max_wait_ns, ~50 us): if it does not show up the
//     launch pair does nothing (or only publishes) and the daemon simply enqueues the next
//     pair -- no kernel ever spins for long, no host synchronisation per poll;
//   * a rank only STARTS a round while it has budget (rounds per applied gradient) and gossip
//     is enabled; a round whose snapshot is already out is always completed.
// host_fb (pinned, optional): [0] = decided bits, [1] = rounds completed, [2] = status word.
// ---------------------------------------------------------------------------
__global__ void sgp_bilat_decide_kernel(const SgpArgs a, const int pub_grid, const int passive,
                                        const unsigned long long max_wait_ns, uint32_t* host_fb)
{
    __shared__ int s_all, s_stop;
    __shared__ uint32_t s_published, s_may_start;
    SgpState* st = a.st;
    const uint32_t step = *((volatile uint32_t*)&st->step);
    RowInfo row;
    load_row(a, step, row);
    int segs = a.segments < 1 ? 1 : a.segments;
    if (segs > SGP_SEQ_STRIDE - 1) segs = SGP_SEQ_STRIDE - 1;
    const uint32_t want = step * (uint32_t)SGP_SEQ_STRIDE + (uint32_t)segs;
    // bilat_budget / bilat_enabled are rewritten asynchronously (sgp_bilat_ctl_kernel on the
    // training stream): ONE thread samples them and the whole CTA uses that sample, so that every
    // thread takes the same branch around the barrier loop below
    if (threadIdx.x == 0) {
        s_published = *((volatile uint32_t*)&st->bilat_published);
        s_may_start = ((*((volatile uint32_t*)&st->bilat_enabled) != 0u) &&
                       (*((volatile uint32_t*)&st->bilat_budget) != 0u)) ? 1u : 0u;
    }
    __syncthreads();
    const uint32_t published = s_published;
    const bool may_start = s_may_start != 0u;
    const bool engaged = published != 0u || may_start;

    int ready = 0;
    if (engaged) {
        const unsigned long long t0 = globaltimer_ns();
        while (true) {
            if (threadIdx.x == 0) s_all = 1;
            __syncthreads();
            for (int k = 0; k < row.n_in; ++k) {
                const int j = row.in[k];
                if (j < 0) continue;
                for (int f = threadIdx.x; f < pub_grid; f += blockDim.x)
                    if ((int32_t)(ld_acquire_sys(&a.pads[j]->pub_seq[f]) - want) < 0) s_all = 0;
            }
            __syncthreads();
            // ONE thread decides whether to stop (the deadline must not be evaluated per thread:
            // threads straddling it would leave the barrier loop at different iterations)
            if (threadIdx.x == 0) s_stop = (s_all != 0) || (globaltimer_ns() - t0 > max_wait_ns);
            __syncthreads();
            ready = s_all;
            const int stop = s_stop;
            __syncthreads();                  // s_all / s_stop are rewritten by the next iteration
            if (stop) break;
            __nanosleep(500);
        }
    }
    if (threadIdx.x != 0) return;
    uint32_t acks_ok = 1u;
    if (step >= st->ack_from + 2u) {
        RowInfo prev;
        load_row(a, step - 2u, prev);
        for (int k = 0; k < prev.n_out; ++k) {
            const int o = prev.out[k];
            if (o < 0 || o == a.rank) continue;
            if ((int32_t)(ld_acquire_sys(&a.pads[a.rank]->ack_seq[o]) - (step - 1u)) < 0) acks_ok = 0u;
        }
    }
    const bool do_publish = !published && may_start && acks_ok && (ready || !passive);
    const bool do_pull = ready && (published || do_publish);
    uint32_t cmd = 0u;
    if (do_publish && do_pull)
        cmd = SGP_F_PHASE1 | SGP_F_PUBLISH | SGP_F_KEEP_Z | SGP_F_PHASE2 | SGP_F_SELF_FROM_Z;
    else if (do_publish)
        cmd = SGP_F_PHASE1 | SGP_F_PUBLISH | SGP_F_KEEP_Z | SGP_F_NO_ROTATE;
    else if (do_pull)
        cmd = SGP_F_PHASE2 | SGP_F_PUBLISH | SGP_F_SELF_FROM_Z;
    if (do_publish) {                          // starting a round consumes budget
        // (compare-and-swap: a budget that sgp_bilat_ctl_kernel rewrote in the meantime wins)
        const uint32_t bud = *((volatile uint32_t*)&st->bilat_budget);
        if (bud != 0xFFFFFFFFu && bud > 0u) atomicCAS(&st->bilat_budget, bud, bud - 1u);
    }
    st->bilat_cmd = cmd;
    st->bilat_done = (uint32_t)ready;
    __threadfence();
    if (host_fb) {
        ((volatile uint32_t*)host_fb)[0] = cmd;
        ((volatile uint32_t*)host_fb)[1] = st->bilat_round + (do_pull ? 1u : 0u);
        ((volatile uint32_t*)host_fb)[2] = st->status;
        __threadfence_system();
    }
}

// budget < 0 / enabled < 0: leave the field alone.  budget == INT_MAX: unbounded
__global__ void sgp_bilat_ctl_kernel(SgpState* st, int budget, int enabled)
{
    if (budget >= 0) st->bilat_budget = (budget == 0x7FFFFFFF) ? 0xFFFFFFFFu : (uint32_t)budget;
    if (enabled >= 0) st->bilat_enabled = (uint32_t)enabled;
    __threadfence();
}

// ---------------------------------------------------------------------------
// AR-SGD comparator: one-shot P2P all-reduce of the (symmetric) gradient
// buffers fused with the SGD update.  Every rank sums in rank order, so the
// replicas stay bit-identical.  pub_seq doubles as the "gradients ready"
// barrier, ack_seq as the "done reading" barrier.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(SGP_THREADS, 2)
sgp_allreduce_sgd_kernel(const SgpArgs a, void* const* grad_peers)
{
    __shared__ int s_ok;
    SgpState* st = a.st;
    const uint32_t step = *((volatile uint32_t*)&st->step);
    const int tid = threadIdx.x, b = blockIdx.x;
    const uint32_t flags = a.flags;
    const long long nchunks = a.n / SGP_CHUNK;
    SgpSignalPad* mypad = a.pads[a.rank];
    const SgpHyper hp = *a.hyper;
    const uint64_t pol_first = l2_evict_first_policy();

    // gradients of this rank were produced by earlier kernels on this stream
    if (tid == 0) {
        s_ok = 1;
        __threadfence_system();
        st_release_sys(&mypad->pub_seq[b], step + 1u);
    }
    __syncthreads();
    if (tid < a.world && tid != a.rank)
        if (!spin_wait_geq(&a.pads[tid]->pub_seq[b], step + 1u, st, a.timeout_ns,
                           SGP_ERR_TIMEOUT_PUB))
            s_ok = 0;
    __syncthreads();

    if (s_ok) {
        const float inv_world = hp.grad_scale / (float)a.world;
        for (long long c = b; c < nchunks; c += gridDim.x) {
            const long long base = c * SGP_CHUNK + (long long)tid * SGP_VEC;
            float4 acc[SGP_UNROLL];
#pragma unroll
            for (int u = 0; u < SGP_UNROLL; ++u) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int r = 0; r < a.world; ++r) {
                float4 gv[SGP_UNROLL];
#pragma unroll
                for (int u = 0; u < SGP_UNROLL; ++u) {
                    const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                    if (flags & SGP_F_GRAD_BF16) {
                        uint2 raw;
                        const uint2* p = reinterpret_cast<const uint2*>(
                            reinterpret_cast<const __nv_bfloat16*>(grad_peers[r]) + i);
                        asm volatile("ld.global.L1::no_allocate.v2.u32 {%0,%1}, [%2];"
                                     : "=r"(raw.x), "=r"(raw.y) : "l"(p));
                        gv[u] = bf16x4_to_f4(raw);
                    } else {
                        gv[u] = ld_stream_f4(reinterpret_cast<const float4*>(
                            reinterpret_cast<const float*>(grad_peers[r]) + i));
                    }
                }
#pragma unroll
                for (int u = 0; u < SGP_UNROLL; ++u) {
                    acc[u].x += gv[u].x; acc[u].y += gv[u].y;
                    acc[u].z += gv[u].z; acc[u].w += gv[u].w;
                }
            }
#pragma unroll
            for (int u = 0; u < SGP_UNROLL; ++u) {
                const long long i = base + (long long)u * SGP_THREADS * SGP_VEC;
                float4 xv = ld_once_f4(reinterpret_cast<const float4*>(a.z + i), pol_first);
                float4 mv = ld_once_f4(reinterpret_cast<const float4*>(a.m + i), pol_first);
                const float4 gv = mul4(acc[u], inv_world);
                sgd1(xv.x, gv.x, mv.x, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                sgd1(xv.y, gv.y, mv.y, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                sgd1(xv.z, gv.z, mv.z, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                sgd1(xv.w, gv.w, mv.w, hp.lr, hp.momentum, hp.weight_decay, hp.nesterov);
                st_f4(reinterpret_cast<float4*>(a.m + i), mv);
                st_f4(reinterpret_cast<float4*>(a.z + i), xv);
                if (flags & SGP_F_SHADOW)
                    st_u2(reinterpret_cast<uint2*>(a.shadow + i), f4_to_bf16x4(xv));
            }
        }
    }

    __syncthreads();
    if (tid == 0 && cta_done_is_last(st)) {
        // tell every peer we are done with its gradients, then wait until every
        // peer is done with ours (the next backward overwrites them)
        for (int r = 0; r < a.world; ++r)
            if (r != a.rank) st_release_sys(&a.pads[r]->ack_seq[a.rank], step + 1u);
        for (int r = 0; r < a.world; ++r)
            if (r != a.rank)
                spin_wait_geq(&mypad->ack_seq[r], step + 1u, st, a.timeout_ns, SGP_ERR_TIMEOUT_ACK);
        *((volatile uint32_t*)&st->done_ctas) = 0u;
        *((volatile uint32_t*)&st->step) = step + 1u;
        __threadfence();
    }
}

// after the all-reduce the caller's gradient buffer is cleared by this rank
__global__ void __launch_bounds__(SGP_THREADS)
sgp_zero_kernel(float4* p, long long n16)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n16;
         i += (long long)gridDim.x * blockDim.x)
        p[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// ---------------------------------------------------------------------------
// Device barrier across ranks (model.block())
// ---------------------------------------------------------------------------
__global__ void sgp_barrier_kernel(SgpSignalPad* const* pads, SgpState* st, int rank, int world,
                                   unsigned long long timeout_ns)
{
    const uint32_t epoch = st->bar_epoch + 1u;
    const int t = threadIdx.x;
    __threadfence_system();
    if (t < world) st_release_sys(&pads[t]->bar_seq[rank], epoch);   // tell everyone
    if (t < world)
        spin_wait_geq(&pads[rank]->bar_seq[t], epoch, st, timeout_ns, SGP_ERR_TIMEOUT_BAR);
    __syncthreads();
    if (t == 0) { st->bar_epoch = epoch; __threadfence(); }
}

// ---------------------------------------------------------------------------
// x *= s  or  x /= s  over a flat buffer (ps_numerator / unbias parity path)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(SGP_THREADS)
sgp_scale_kernel(float* x, long long n, const float* scalar, int invert, __nv_bfloat16* shadow)
{
    const float s = invert ? (1.f / *scalar) : *scalar;
    const long long n4 = n / 4;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4;
         i += (long long)gridDim.x * blockDim.x) {
        float4 v = reinterpret_cast<float4*>(x)[i];
        v = mul4(v, s);
        reinterpret_cast<float4*>(x)[i] = v;
        if (shadow) reinterpret_cast<uint2*>(shadow)[i] = f4_to_bf16x4(v);
    }
}

// ---------------------------------------------------------------------------
// dst = scale * sum_k srcs[k]   over flat fp32 buffers that may live on PEER devices of the same
// process (single-process multi-GPU replicas): the reference's reduce_add_coalesced
// (gossip/distributed.py:523-549, N10) as one kernel of 16-byte P2P loads on the master GPU.
// ---------------------------------------------------------------------------
struct SgpPtrList { const float* p[SGP_MAX_RANKS]; int n; };

__global__ void __launch_bounds__(SGP_THREADS)
sgp_peer_reduce_kernel(float* __restrict__ dst, const SgpPtrList srcs, long long n4, float scale)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4;
         i += (long long)gridDim.x * blockDim.x) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int k = 0; k < srcs.n; ++k) {
            const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(srcs.p[k]) + i);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        reinterpret_cast<float4*>(dst)[i] = mul4(acc, scale);
    }
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
extern "C" {

cudaError_t sgp_launch_step(const SgpArgs* args, int grid, cudaStream_t stream)
{
    sgp_step_kernel<<<grid, SGP_THREADS, 0, stream>>>(*args);
    return cudaGetLastError();
}

cudaError_t sgp_launch_step_pipe(const SgpArgs* args, int grid, cudaStream_t stream)
{
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(sgp_step_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             PIPE_SMEM);
        if (e != cudaSuccess) return e;
        // two CTAs x 64 KB per SM: ask for the large shared-memory carve-out (the default one fits
        // a single CTA: launch__occupancy_limit_shared_mem = 1 in the first ncu capture)
        e = cudaFuncSetAttribute(sgp_step_pipe_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) configured[dev] = true;
    }
    sgp_step_pipe_kernel<<<grid, PIPE_THREADS, PIPE_SMEM, stream>>>(*args);
    return cudaGetLastError();
}

// co-resident CTAs of the pipelined step kernel (dynamic shared memory bound)
int sgp_max_resident_ctas_pipe(int device)
{
    int sms = 0, per_sm = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return 0;
    cudaFuncSetAttribute(sgp_step_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PIPE_SMEM);
    cudaFuncSetAttribute(sgp_step_pipe_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                         cudaSharedmemCarveoutMaxShared);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sgp_step_pipe_kernel, PIPE_THREADS, PIPE_SMEM)
        != cudaSuccess) return 0;
    return sms * per_sm;
}

cudaError_t sgp_launch_gather(const SgpArgs* args, int grid, int pub_grid, cudaStream_t stream)
{
    sgp_gather_kernel<<<grid, SGP_THREADS, 0, stream>>>(*args, pub_grid);
    return cudaGetLastError();
}

cudaError_t sgp_launch_gather_tma(const SgpArgs* args, int grid, int pub_grid, cudaStream_t stream)
{
    const int smem = SGP_TMA_STAGES * SGP_TMA_BYTES + SGP_TMA_STAGES * 8 + 64;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(sgp_gather_tma_kernel,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    sgp_gather_tma_kernel<<<grid, SGP_THREADS, smem, stream>>>(*args, pub_grid);
    return cudaGetLastError();
}

cudaError_t sgp_launch_probe(const SgpArgs* args, int pub_grid, uint32_t* host_flag,
                             cudaStream_t stream)
{
    sgp_probe_kernel<<<1, SGP_THREADS, 0, stream>>>(*args, pub_grid, host_flag);
    return cudaGetLastError();
}

cudaError_t sgp_launch_gather_wait(const SgpArgs* args, int pub_grid, cudaStream_t stream)
{
    sgp_gather_wait_kernel<<<1, SGP_THREADS, 0, stream>>>(*args, pub_grid);
    return cudaGetLastError();
}

cudaError_t sgp_launch_gather_ack(const SgpArgs* args, cudaStream_t stream)
{
    sgp_gather_ack_kernel<<<1, 1, 0, stream>>>(*args);
    return cudaGetLastError();
}

cudaError_t sgp_launch_bilat_decide(const SgpArgs* args, int pub_grid, int passive,
                                    unsigned long long max_wait_ns, uint32_t* host_fb, cudaStream_t stream)
{
    sgp_bilat_decide_kernel<<<1, SGP_THREADS, 0, stream>>>(*args, pub_grid, passive, max_wait_ns, host_fb);
    return cudaGetLastError();
}

cudaError_t sgp_launch_bilat_ctl(SgpState* st, int budget, int enabled, cudaStream_t stream)
{
    sgp_bilat_ctl_kernel<<<1, 1, 0, stream>>>(st, budget, enabled);
    return cudaGetLastError();
}

cudaError_t sgp_launch_allreduce_sgd(const SgpArgs* args, void* const* grad_peers, int grid,
                                     cudaStream_t stream)
{
    sgp_allreduce_sgd_kernel<<<grid, SGP_THREADS, 0, stream>>>(*args, grad_peers);
    return cudaGetLastError();
}

cudaError_t sgp_launch_peer_reduce(float* dst, const float* const* srcs, int nsrc, long long n, float scale,
                                   cudaStream_t stream)
{
    if (nsrc < 1 || nsrc > SGP_MAX_RANKS || (n & 3)) return cudaErrorInvalidValue;
    SgpPtrList l;
    l.n = nsrc;
    for (int k = 0; k < nsrc; ++k) l.p[k] = srcs[k];
    const long long n4 = n / 4;
    int grid = (int)((n4 + SGP_THREADS - 1) / SGP_THREADS);
    if (grid > 148 * 8) grid = 148 * 8;
    if (grid < 1) grid = 1;
    sgp_peer_reduce_kernel<<<grid, SGP_THREADS, 0, stream>>>(dst, l, n4, scale);
    return cudaGetLastError();
}

cudaError_t sgp_launch_zero(void* p, long long bytes, cudaStream_t stream)
{
    const long long n16 = bytes / 16;
    int grid = (int)((n16 + SGP_THREADS - 1) / SGP_THREADS);
    if (grid > 148 * 8) grid = 148 * 8;
    if (grid < 1) grid = 1;
    sgp_zero_kernel<<<grid, SGP_THREADS, 0, stream>>>(reinterpret_cast<float4*>(p), n16);
    return cudaGetLastError();
}

cudaError_t sgp_launch_barrier(SgpSignalPad* const* pads, SgpState* st, int rank, int world,
                               unsigned long long timeout_ns, cudaStream_t stream)
{
    sgp_barrier_kernel<<<1, SGP_MAX_RANKS, 0, stream>>>(pads, st, rank, world, timeout_ns);
    return cudaGetLastError();
}

cudaError_t sgp_launch_scale(float* x, long long n, const float* scalar, int invert,
                             __nv_bfloat16* shadow, cudaStream_t stream)
{
    long long n4 = n / 4;
    int grid = (int)((n4 + SGP_THREADS - 1) / SGP_THREADS);
    if (grid > 148 * 8) grid = 148 * 8;
    if (grid < 1) grid = 1;
    sgp_scale_kernel<<<grid, SGP_THREADS, 0, stream>>>(x, n, scalar, invert, shadow);
    return cudaGetLastError();
}

int sgp_max_resident_ctas(int device)
{
    int sms = 0, per_sm = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sgp_step_kernel, SGP_THREADS, 0)
        != cudaSuccess) return 0;
    return sms * per_sm;
}

// With CUDA's lazy loading (the default) a kernel is loaded at its first launch, and that load may
// have to synchronise the context.  The gossip kernels spin on flags released by other launches: the
// first launch of sgp_gather_ack_kernel, for instance, is queued while sgp_gather_wait_kernel spins
// for the in-neighbour, and with several ranks on one host thread (LocalWorld) that in-neighbour's
// publish is launched only afterwards -- the load would wait for the spin and the spin for the
// launch, until the heartbeat fires.  Loading every gossip kernel of the current device up front
// keeps first launches from waiting on the device.
cudaError_t sgp_preload_kernels()
{
    typedef CUresult (*FuncLoad)(CUfunction);
    static FuncLoad func_load = nullptr;
    if (func_load == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t e = cudaGetDriverEntryPoint("cuFuncLoad", &p, cudaEnableDefault, &q);
        if (e != cudaSuccess) return e;
        if (q != cudaDriverEntryPointSuccess || p == nullptr) return cudaErrorNotSupported;
        func_load = reinterpret_cast<FuncLoad>(p);
    }
    const void* kernels[] = {
        (const void*)sgp_step_kernel, (const void*)sgp_step_pipe_kernel, (const void*)sgp_gather_kernel,
        (const void*)sgp_gather_tma_kernel, (const void*)sgp_probe_kernel, (const void*)sgp_gather_wait_kernel,
        (const void*)sgp_gather_ack_kernel, (const void*)sgp_bilat_decide_kernel,
        (const void*)sgp_bilat_ctl_kernel, (const void*)sgp_allreduce_sgd_kernel, (const void*)sgp_zero_kernel,
        (const void*)sgp_scale_kernel, (const void*)sgp_peer_reduce_kernel, (const void*)sgp_barrier_kernel,
    };
    for (const void* k : kernels) {
        cudaFunction_t f = nullptr;
        cudaError_t e = cudaGetFuncBySymbol(&f, k);
        if (e != cudaSuccess) return e;
        if (func_load(reinterpret_cast<CUfunction>(f)) != CUDA_SUCCESS) return cudaErrorInitializationError;
    }
    return cudaSuccess;
}

}  // extern "C"
