// Persistent rollout kernel: T env steps of ALL co-located actors in ONE launch.
//
// The per-step launch sequence (policy forward -> sample -> env step -> window staging) is bound by fixed costs:
// every launch re-fetches the policy weights from L2 (a chain of dependent round trips, profiles/r01c) and pays
// launch + drain; 128 steps x 3 launches cost ~4.3 ms per rollout for ~0.2 ms of arithmetic.  Actors are
// independent of one another, so the loop over time can move INSIDE the kernel:
//   * a thread-block cluster of 4 CTAs owns 32 actors for the whole chunk;
//   * each CTA keeps a QUARTER of every hidden layer's weights resident in shared memory for all T steps (fetched
//     once with cp.async) and computes that quarter of the layer's columns for the cluster's 32 rows (fp32, packed
//     fma.rn.f32x2); layer outputs reach the CTAs that need them through distributed shared memory;
//   * WARP SPECIALISATION: warps 0..7 ("math warps") run the two hidden layers while warps 8..15 ("env warps") do the
//     half of the SAME env step that does not depend on the action (Philox + Box-Muller draws, Ws.s, |s|^2) -- it
//     depends only on the state at the top of the step, so it stays off the serial chain;
//   * the three exchanges of a step (hidden layer 1 to all peers, last hidden layer rows to their owner, next input
//     tile to all peers) are st.async stores that signal the consumer's mbarrier, not cluster barriers; the cyclic data
//     dependence of a step makes "buffer free" signals unnecessary;
//   * the head runs on all 16 warps (k slices of the last hidden layer for all 8 owned actors); then each CTA finishes
//     ITS 8 actors -- sampling, environment step, window staging -- one warp per actor; observations / env state never
//     leave shared memory between steps;
//   * finished windows go to a per-actor outbox with their completion step; sb200_ppo_rollout_commit_f32 assigns
//     FIFO slots in the reference's (step, actor) arrival order afterwards and copies them into the replay ring.
// The schedule follows clock64 traces of the kernel (tools/rollout_trace.py, profiles/r02b_rollout_trace_*).
// Sampling and environment arithmetic (and their Philox keys) are those of rollout.cu, so both paths draw the
// same noise; the policy forward is fp32 FMA (the per-step path uses 3xTF32 tensor-core products; both are
// fp32-accurate, they differ by rounding order only).
#include <cooperative_groups.h>

#include <algorithm>

#include "common.cuh"
#include "rollout_dev.cuh"

namespace {

namespace cg = cooperative_groups;

constexpr int RF_CS = 4;            // CTAs per cluster
constexpr int RF_ROWS = 32;         // actors per cluster
constexpr int RF_OWN = RF_ROWS / RF_CS;
constexpr int RF_THREADS = 512;     // 16 warps: 8 math warps, 8 env warps

// -DRF_TRACE (tools/rollout_trace.py builds that variant; never the shipped library): clock64 stamps of cluster 0's
// first steps, one row per (CTA, step), read back through sb200_debug_rf_trace().
// RF_TID: the thread index the stamps and the layer functions go by
#define RF_TID threadIdx.x
#ifdef RF_TRACE
constexpr int RF_TR_STEPS = 8, RF_TR_IDS = 32;
__device__ long long g_rf_trace[RF_CS][RF_TR_STEPS][RF_TR_IDS];
#define RF_STAMP(id, who)                                                                           \
    do {                                                                                            \
        if (blockIdx.x < RF_CS && RF_TID == (who) && rf_t >= 2 && rf_t < 2 + RF_TR_STEPS)           \
            g_rf_trace[blockIdx.x][rf_t - 2][id] = clock64();                                       \
    } while (0)
#else
#define RF_STAMP(id, who) do { } while (0)
#endif

struct RfParams {
    const float* W[3];
    const float* b[3];
    int ldw[3];
    int act[3];
    int D, H1, H2, A;
    const float* zf;
    float zf_eps;
    const float* log_var;
    const float* log_noise;
    unsigned long long agent_seed;
    int deterministic;
    float* state;
    const float* WsT;
    const float* WaT;
    int* ep_step;
    int max_steps;
    unsigned long long env_seed;
    float* action;
    float* pd;
    float* obs_next;
    float* reward;
    float* done;
    int* stage_pos;
    float* stage_obs;
    float* stage_act;
    float* stage_pd;
    float* stage_rew;
    float* stage_done;
    float* o_obs;
    float* o_act;
    float* o_pd;
    float* o_rew;
    float* o_done;
    int* ev_step;
    int* ev_count;
    int Wout;                       // outbox entries per actor
    int N, n_step, stride, T;
    const unsigned long long* step_ctr;
    // shared-memory plan (float offsets)
    int oW1, oW2, oWh, oB, oX0, oH1, oH2, oPart, oZf, oEnv, oS, oNext, oAct, oPre;
    int ldx0, ldh1, ldh2;
};

__device__ __forceinline__ float rf_act(float v, int act) {
    if (act == SB200_ACT_RELU) return fmaxf(v, 0.0f);
    if (act == SB200_ACT_TANH) return tanhf(v);
    return v;
}

__device__ __forceinline__ unsigned rf_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned rf_mapa(unsigned addr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void rf_bar_math() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// ---- mbarrier-signalled DSMEM hand-off.  st.async carries the data AND the completion count to the consumer's
// mbarrier, so the producer needs no fence and the consumer polls its own shared memory.  (barrier.cluster.arrive.release
// would compile to MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR in front of the barrier -- the kernel's global stores of the step
// must drain to L2 first -- and the wait to a CCTL.IVALL: three times per env step.)
__device__ __forceinline__ void rf_mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(rf_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void rf_mbar_arm(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(rf_smem_u32(bar)), "r"(bytes) : "memory");
}
// spin until the phase with this parity has completed; a transaction count that can never be met would hang the GPU, so
// the spin is bounded (~1 s) and traps instead
__device__ __forceinline__ void rf_mbar_wait(unsigned long long* bar, unsigned parity) {
    const unsigned a = rf_smem_u32(bar);
    for (unsigned spin = 0;; ++spin) {
        unsigned ok;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(a), "r"(parity) : "memory");
        if (ok) return;
        if (spin > (1u << 26)) __trap();
    }
}
__device__ __forceinline__ void rf_st_async_v4(unsigned dst_cluster_addr, const float4& v, unsigned mbar_cluster_addr) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(dst_cluster_addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"(mbar_cluster_addr) : "memory");
}

// The last hidden layer on the 8 math warps (tid 0..255), this CTA's Nc columns for the cluster's 32 rows; each row goes
// only to the CTA that owns the actor, into its Hout [8][ldout] (input of the head).  Xin [32][ldin] and Ws [K][Nc] live
// in shared memory; K % 4 == 0.
//   warp = (row group rg = warp & 3: rows 8rg..8rg+7, k quarter pair), lane = (column quad, k half) -> 4-way k split,
//   partial tiles summed in a fixed order (deterministic) through Part [4][32][Nc].  8 x 4 register tiles: 12 LDS.128 per
//   128 FMA -- the layer loop is bound by shared-memory loads, not by FMA issue -- and the activation loads of a warp
//   (ONE 8-row group) are warp-wide broadcasts.  Packed fma.rn.f32x2: each half is an IEEE fma, so the result is that
//   of two scalar fmaf; it only halves the issue slots.
__device__ __forceinline__ void rf2_layer(const float* __restrict__ Xin, int ldin, int K, const float* __restrict__ Ws,
                                          int Nc, const float* __restrict__ bias_s, int act, float* __restrict__ Hout,
                                          int ldout, int col0, float* __restrict__ Part, unsigned smem_base,
                                          unsigned crank, int rf_t, unsigned bar_off) {
    const int tid = (int)RF_TID, warp = tid >> 5, lane = tid & 31;
    const int rg = warp & 3, ks = ((warp >> 2) << 1) | (lane >> 4), cg0 = lane & 15;
    const int kq = (((K >> 2) + 3) >> 2) << 2;               // k span of one split (multiple of 4)
    const int k_lo = ks * kq, k_hi = min(K, k_lo + kq);
    const int nq = Nc >> 2;
    const float* xr = Xin + (rg * 8) * ldin;
    for (int c4 = cg0; c4 < nq; c4 += 16) {
        const float* wp = Ws + c4 * 4;
        float2 acc[8][2];
#pragma unroll
        for (int r = 0; r < 8; ++r) acc[r][0] = acc[r][1] = make_float2(0.0f, 0.0f);
#pragma unroll 2
        for (int k = k_lo; k < k_hi; k += 4) {
            const float4 w0 = *reinterpret_cast<const float4*>(wp + (k + 0) * Nc);
            const float4 w1 = *reinterpret_cast<const float4*>(wp + (k + 1) * Nc);
            const float4 w2 = *reinterpret_cast<const float4*>(wp + (k + 2) * Nc);
            const float4 w3 = *reinterpret_cast<const float4*>(wp + (k + 3) * Nc);
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const float4 a = *reinterpret_cast<const float4*>(xr + r * ldin + k);
                float2 aa = make_float2(a.x, a.x);
                acc[r][0] = __ffma2_rn(aa, make_float2(w0.x, w0.y), acc[r][0]);
                acc[r][1] = __ffma2_rn(aa, make_float2(w0.z, w0.w), acc[r][1]);
                aa = make_float2(a.y, a.y);
                acc[r][0] = __ffma2_rn(aa, make_float2(w1.x, w1.y), acc[r][0]);
                acc[r][1] = __ffma2_rn(aa, make_float2(w1.z, w1.w), acc[r][1]);
                aa = make_float2(a.z, a.z);
                acc[r][0] = __ffma2_rn(aa, make_float2(w2.x, w2.y), acc[r][0]);
                acc[r][1] = __ffma2_rn(aa, make_float2(w2.z, w2.w), acc[r][1]);
                aa = make_float2(a.w, a.w);
                acc[r][0] = __ffma2_rn(aa, make_float2(w3.x, w3.y), acc[r][0]);
                acc[r][1] = __ffma2_rn(aa, make_float2(w3.z, w3.w), acc[r][1]);
            }
        }
#pragma unroll
        for (int r = 0; r < 8; ++r)
            *reinterpret_cast<float4*>(Part + ((ks * RF_ROWS + rg * 8 + r) * Nc + c4 * 4)) =
                make_float4(acc[r][0].x, acc[r][0].y, acc[r][1].x, acc[r][1].y);
    }
    RF_STAMP(5, 0);
    rf_bar_math();
    RF_STAMP(6, 0);
    for (int idx = tid; idx < RF_ROWS * nq; idx += 256) {
        const int row = idx / nq, c4 = idx - row * nq;
        const float* pp = Part + row * Nc + c4 * 4;
        const float4 p0 = *reinterpret_cast<const float4*>(pp);
        const float4 p1 = *reinterpret_cast<const float4*>(pp + RF_ROWS * Nc);
        const float4 p2 = *reinterpret_cast<const float4*>(pp + 2 * RF_ROWS * Nc);
        const float4 p3 = *reinterpret_cast<const float4*>(pp + 3 * RF_ROWS * Nc);
        const float4 bv = *reinterpret_cast<const float4*>(bias_s + c4 * 4);
        float4 o;
        o.x = rf_act(((p0.x + p1.x) + (p2.x + p3.x)) + bv.x, act);
        o.y = rf_act(((p0.y + p1.y) + (p2.y + p3.y)) + bv.y, act);
        o.z = rf_act(((p0.z + p1.z) + (p2.z + p3.z)) + bv.z, act);
        o.w = rf_act(((p0.w + p1.w) + (p2.w + p3.w)) + bv.w, act);
        const unsigned owner = (unsigned)(row / RF_OWN);
        float* qd = Hout + (row - (int)owner * RF_OWN) * ldout + col0 + c4 * 4;
        if (owner == crank) {
            *reinterpret_cast<float4*>(qd) = o;
        } else {
            const unsigned pb = rf_mapa(smem_base, owner);
            rf_st_async_v4(pb + (rf_smem_u32(qd) - smem_base), o, pb + bar_off);
        }
    }
}

// First hidden layer on the 8 math warps WITHOUT a shared-memory reduction: K = D is short (64), so the 4-way k split of
// rf2_layer would spend more on partial tiles, the barrier and the second pass (1.5 K cycles) than on its 4 k quads of
// FMAs.  Warp w owns rows 4w..4w+3, lane = (column quad, k half); the two k halves of a lane pair are summed by shuffle
// (each lane keeps two of the four rows) and the epilogue stores / pushes the result into every CTA's copy of
// Hout [32][ldout] straight from registers.
__device__ __forceinline__ void rf2_layer1(const float* __restrict__ Xin, int ldin, int K, const float* __restrict__ Ws, int Nc,
                                           const float* __restrict__ bias_s, int act, float* __restrict__ Hout, int ldout,
                                           int col0, unsigned smem_base, unsigned crank, unsigned bar_off) {
    const int tid = (int)RF_TID, warp = tid >> 5, lane = tid & 31;
    const int cg0 = lane & 15, kh = lane >> 4;
    const bool up = kh != 0;
    const int kq = (((K >> 2) + 1) >> 1) << 2;               // k span of one half (multiple of 4)
    const int k_lo = kh * kq, k_hi = min(K, k_lo + kq);
    const int nq = Nc >> 2;
    const float* xr = Xin + (warp * 4) * ldin;
    unsigned pb[RF_CS - 1];
#pragma unroll
    for (int c = 1; c < RF_CS; ++c) pb[c - 1] = rf_mapa(smem_base, (crank + (unsigned)c) % RF_CS);
    for (int c4 = cg0; c4 < ((nq + 15) & ~15); c4 += 16) {    // uniform trip count: the shuffles need the whole warp
        const bool on = c4 < nq;
        const float* wp = Ws + (on ? c4 : 0) * 4;
        float2 acc[4][2];
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[r][0] = acc[r][1] = make_float2(0.0f, 0.0f);
#pragma unroll 2
        for (int k = k_lo; k < k_hi; k += 4) {
            const float4 w0 = *reinterpret_cast<const float4*>(wp + (k + 0) * Nc);
            const float4 w1 = *reinterpret_cast<const float4*>(wp + (k + 1) * Nc);
            const float4 w2 = *reinterpret_cast<const float4*>(wp + (k + 2) * Nc);
            const float4 w3 = *reinterpret_cast<const float4*>(wp + (k + 3) * Nc);
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float4 a = *reinterpret_cast<const float4*>(xr + r * ldin + k);
                float2 aa = make_float2(a.x, a.x);
                acc[r][0] = __ffma2_rn(aa, make_float2(w0.x, w0.y), acc[r][0]);
                acc[r][1] = __ffma2_rn(aa, make_float2(w0.z, w0.w), acc[r][1]);
                aa = make_float2(a.y, a.y);
                acc[r][0] = __ffma2_rn(aa, make_float2(w1.x, w1.y), acc[r][0]);
                acc[r][1] = __ffma2_rn(aa, make_float2(w1.z, w1.w), acc[r][1]);
                aa = make_float2(a.z, a.z);
                acc[r][0] = __ffma2_rn(aa, make_float2(w2.x, w2.y), acc[r][0]);
                acc[r][1] = __ffma2_rn(aa, make_float2(w2.z, w2.w), acc[r][1]);
                aa = make_float2(a.w, a.w);
                acc[r][0] = __ffma2_rn(aa, make_float2(w3.x, w3.y), acc[r][0]);
                acc[r][1] = __ffma2_rn(aa, make_float2(w3.z, w3.w), acc[r][1]);
            }
        }
        const float4 bv = *reinterpret_cast<const float4*>(bias_s + (on ? c4 : 0) * 4);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const float2 s0 = up ? acc[r][0] : acc[r + 2][0], s1 = up ? acc[r][1] : acc[r + 2][1];
            const float2 m0 = up ? acc[r + 2][0] : acc[r][0], m1 = up ? acc[r + 2][1] : acc[r][1];
            float4 o;
            o.x = rf_act((m0.x + __shfl_xor_sync(0xffffffffu, s0.x, 16)) + bv.x, act);
            o.y = rf_act((m0.y + __shfl_xor_sync(0xffffffffu, s0.y, 16)) + bv.y, act);
            o.z = rf_act((m1.x + __shfl_xor_sync(0xffffffffu, s1.x, 16)) + bv.z, act);
            o.w = rf_act((m1.y + __shfl_xor_sync(0xffffffffu, s1.y, 16)) + bv.w, act);
            if (on) {
                const int row = warp * 4 + (up ? 2 : 0) + r;
                float* qd = Hout + row * ldout + col0 + c4 * 4;
                *reinterpret_cast<float4*>(qd) = o;
                const unsigned off = rf_smem_u32(qd) - smem_base;
#pragma unroll
                for (int c = 0; c < RF_CS - 1; ++c) rf_st_async_v4(pb[c] + off, o, pb[c] + bar_off);
            }
        }
    }
}

__global__ void __cluster_dims__(RF_CS, 1, 1) __launch_bounds__(RF_THREADS, 1)
    ppo_rollout2_kernel(const __grid_constant__ RfParams p) {
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned crank = cluster.block_rank();
    extern __shared__ __align__(16) float smem[];
    const unsigned smem_base = rf_smem_u32(smem);
    unsigned peer_base[RF_CS - 1];
#pragma unroll
    for (int c = 1; c < RF_CS; ++c) peer_base[c - 1] = rf_mapa(smem_base, (crank + (unsigned)c) % RF_CS);
    __shared__ int s_pos[RF_OWN], s_ep[RF_OWN], s_cnt[RF_OWN];
    __shared__ __align__(8) unsigned long long s_bar[3];      // hidden layer 1 | last hidden layer rows | next input tile

    // (tried: the two roles on swapped warp halves, in case the scheduler's preference for one end of the warp index range
    // starved the layers -- no difference, profiles/r02b_rollout_trace_*)
    const int tid = (int)RF_TID, lane = tid & 31, warp = tid >> 5;
    const int D = p.D, H1 = p.H1, H2 = p.H2, A = p.A;
    const int Nc1 = H1 / RF_CS, Nc2 = H2 / RF_CS;
    const int ldwh = p.ldw[2];
    float* W1s = smem + p.oW1;          // [D][Nc1]
    float* W2s = smem + p.oW2;          // [H1][Nc2]
    float* Whs = smem + p.oWh;          // [H2][ldwh]
    float* B1s = smem + p.oB;           // [Nc1] | [Nc2] | [ldwh]
    float* B2s = B1s + Nc1;
    float* Bhs = B2s + Nc2;
    float* X0 = smem + p.oX0;           // [32][ldx0]  z-filtered observations of the cluster's actors
    float* Hb1 = smem + p.oH1;          // [32][ldh1]
    float* Hb2 = smem + p.oH2;          // [8][ldh2]   last hidden layer, owned actors only
    float* Part = smem + p.oPart;       // [4][32][max(Nc1, Nc2)] k-split partial tiles | [16][8][ldwh] head slice sums
    float* Zm = smem + p.oZf;           // [D] mean | [D] std
    float* Zs = Zm + D;
    float* EWs = smem + p.oEnv;         // [D][D] | [A][D]   (k-major)
    float* EWa = EWs + D * D;
    float* S = smem + p.oS;             // [8][D]   env state of the owned actors (what they observe next)
    float* Nx = smem + p.oNext;         // [8][D]   true successor of the step
    float* Ac = smem + p.oAct;          // [8][A]   sampled actions | std | N(0,1) draws
    float* Sd = Ac + RF_OWN * A;
    float* Zn = Sd + RF_OWN * A;
    float* Eacc = smem + p.oPre;        // [8][D] Ws.s | [8][D] env noise | [8][D] reset draws | [16] |s|^2, reward noise
    float* Egx = Eacc + RF_OWN * D;
    float* Erz = Egx + RF_OWN * D;
    float* Eq = Erz + RF_OWN * D;
    const long long row0 = (long long)(blockIdx.x / RF_CS) * RF_ROWS;

    // ---- one-time loads: weight slices, biases, env matrices (cp.async burst), z-filter columns, actor state
    for (int f = tid; f < D * (Nc1 >> 2); f += RF_THREADS) {
        const int k = f / (Nc1 >> 2), q = f - k * (Nc1 >> 2);
        cp_async16(W1s + k * Nc1 + q * 4, p.W[0] + (long long)k * p.ldw[0] + crank * Nc1 + q * 4, 16);
    }
    for (int f = tid; f < H1 * (Nc2 >> 2); f += RF_THREADS) {
        const int k = f / (Nc2 >> 2), q = f - k * (Nc2 >> 2);
        cp_async16(W2s + k * Nc2 + q * 4, p.W[1] + (long long)k * p.ldw[1] + crank * Nc2 + q * 4, 16);
    }
    for (int f = tid; f < (H2 * ldwh) >> 2; f += RF_THREADS) cp_async16(Whs + f * 4, p.W[2] + f * 4, 16);
    for (int f = tid; f < (D * D) >> 2; f += RF_THREADS) cp_async16(EWs + f * 4, p.WsT + f * 4, 16);
    for (int f = tid; f < (A * D) >> 2; f += RF_THREADS) cp_async16(EWa + f * 4, p.WaT + f * 4, 16);
    cp_async_commit();
    for (int n = tid; n < Nc1; n += RF_THREADS) B1s[n] = p.b[0][crank * Nc1 + n];
    for (int n = tid; n < Nc2; n += RF_THREADS) B2s[n] = p.b[1][crank * Nc2 + n];
    for (int n = tid; n < ldwh; n += RF_THREADS) Bhs[n] = (n < A) ? p.b[2][n] : 0.0f;
    if (p.zf != nullptr) {
        const float cnt = p.zf[2 * D];
        for (int k = tid; k < D; k += RF_THREADS) {
            const float mean = p.zf[k] / cnt;
            const float var = p.zf[D + k] / cnt - mean * mean;
            Zm[k] = mean;
            Zs[k] = fmaxf(sqrtf(var), p.zf_eps);
        }
    }
    if (tid < RF_OWN) {
        const long long i = row0 + crank * RF_OWN + tid;
        s_pos[tid] = (i < p.N) ? p.stage_pos[i] : 0;
        s_ep[tid] = (i < p.N) ? p.ep_step[i] : 0;
        s_cnt[tid] = 0;
    }
    __syncthreads();
    for (int idx = tid; idx < RF_ROWS * D; idx += RF_THREADS) {       // all 32 rows: every CTA needs the full input
        const int m = idx / D, k = idx - m * D;
        const long long i = row0 + m;
        float v = (i < p.N) ? p.state[i * D + k] : 0.0f;
        const int own = m - (int)crank * RF_OWN;
        if (own >= 0 && own < RF_OWN) S[own * D + k] = v;
        if (p.zf != nullptr) v = fminf(fmaxf((v - Zm[k]) / Zs[k], -5.0f), 5.0f);
        X0[m * p.ldx0 + k] = (i < p.N) ? v : 0.0f;
    }
    const unsigned long long ctr0 = (p.step_ctr != nullptr) ? *p.step_ctr : 0ull;
    if (tid == 0) {
        for (int i = 0; i < 3; ++i) rf_mbar_init(&s_bar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const unsigned bar_off_h1 = rf_smem_u32(&s_bar[0]) - smem_base, bar_off_h2 = rf_smem_u32(&s_bar[1]) - smem_base;
    const unsigned bar_off_x0 = rf_smem_u32(&s_bar[2]) - smem_base;
    // bytes a CTA receives from its three peers per step: their column quarters of hidden layer 1 for all 32 rows, their
    // column quarters of the last hidden layer for the 8 owned rows, their 8 rows of the next input tile (each below the
    // mbarrier's 2^20 transaction limit: rf_plan)
    const unsigned tx_h1 = 3u * RF_ROWS * Nc1 * 4u, tx_h2 = 3u * RF_OWN * Nc2 * 4u, tx_x0 = 3u * RF_OWN * D * 4u;
    cp_async_wait<0>();
    cluster.sync();                                   // weights landed; barriers initialised; every peer is running

    const bool math = warp < RF_OWN;                  // warps 0..7: layers, then owner of actor `warp`
    const int own = warp & (RF_OWN - 1);              // owned actor this warp works for (owner or env warp)
    const bool owner = math;
    const int m_own = (int)crank * RF_OWN + own;
    const long long i_own = row0 + m_own;
    const bool valid = owner && (i_own < p.N);
    {
        const float sc = (i_own < p.N && p.log_noise != nullptr) ? expf(p.log_noise[i_own]) : 1.0f;
        if (owner && lane < A) Sd[own * A + lane] = __fmul_rn(expf(p.log_var[lane]), sc);     // constant over the chunk
    }
    __syncthreads();

    for (int t = 0; t < p.T; ++t) {
        const unsigned long long ctr = ctr0 + (unsigned long long)t;
        const bool final_step = (t == p.T - 1);
        const int rf_t = t;
        RF_STAMP(0, 0);
        if (tid == 0) {                                       // arm this step's phases (the previous ones were consumed)
            rf_mbar_arm(&s_bar[0], tx_h1);
            rf_mbar_arm(&s_bar[1], tx_h2);
        }
        if (math) {
            if (t > 0) {                                      // the input tile: own rows (math warps wrote them) + the peers' rows
                rf_bar_math();
                rf_mbar_wait(&s_bar[2], (unsigned)(t - 1) & 1u);
            }
            RF_STAMP(18, 0);
            if (tid == 0 && !final_step) rf_mbar_arm(&s_bar[2], tx_x0);     // next tile's phase: only now is the previous one complete
            rf2_layer1(X0, p.ldx0, D, W1s, Nc1, B1s, p.act[0], Hb1, p.ldh1, (int)crank * Nc1, smem_base, crank, bar_off_h1);
            RF_STAMP(3, 0);
            rf_bar_math();                                    // hidden layer 1: own columns + the peers' columns
            rf_mbar_wait(&s_bar[0], (unsigned)t & 1u);
            RF_STAMP(4, 0);
            rf2_layer(Hb1, p.ldh1, H1, W2s, Nc2, B2s, p.act[1], Hb2, p.ldh2, (int)crank * Nc2, Part, smem_base, crank, rf_t,
                      bar_off_h2);
            RF_STAMP(7, 0);
        } else {
            // ---- env warp h: everything of this step that does not depend on the action (arithmetic and Philox keys of
            // sample_one() / synth_env_block() in rollout.cu), concurrently with the layers
            RF_STAMP(16, 256);
            const int h = own;
            const long long ih = row0 + (int)crank * RF_OWN + h;
            const float* sh = S + h * D;
            float q = 0.0f;
            for (int d = lane; d < D; d += 32) q += sh[d] * sh[d];
            q = warp_sum(q);
            const bool h_done = (p.max_steps > 0) && (s_ep[h] + 1 >= p.max_steps);
            for (int d = lane; d < D; d += 32) {
                float acc = 0.0f;                              // WsT is [k][d]: conflict-free across lanes
#pragma unroll 8
                for (int k = 0; k < D; ++k) acc = fmaf(EWs[k * D + d], sh[k], acc);
                const Philox4 r = philox4x32_10(p.env_seed ^ 0x5851F42D4C957F2Dull, ctr,
                                                ((unsigned long long)ih << 20) | (unsigned long long)d);
                const float2 gz = box_muller(r.x, r.y);
                Eacc[h * D + d] = acc;
                Egx[h * D + d] = gz.x;
                Erz[h * D + d] = h_done ? box_muller(r.z, r.w).x : 0.0f;
                if (d == 0) {
                    Eq[2 * h] = q;
                    Eq[2 * h + 1] = gz.y;
                }
            }
            if (!p.deterministic && lane < A) {                // PPOAgent.act's N(0,1) draws: keys of sample_one()
                const int j = lane;
                const Philox4 r = philox4x32_10(p.agent_seed, ctr, ((unsigned long long)ih << 16) | (unsigned long long)(j >> 2));
                const float2 z01 = box_muller(r.x, r.y), z23 = box_muller(r.z, r.w);
                const int c = j & 3;
                Zn[h * A + j] = (c == 0) ? z01.x : (c == 1) ? z01.y : (c == 2) ? z23.x : z23.y;
            }
            RF_STAMP(17, 256);
        }
        __syncthreads();                                      // last hidden layer: own columns + the peers' columns
        rf_mbar_wait(&s_bar[1], (unsigned)t & 1u);
        // ---- head: warp w takes the k slice [w H2/16, (w+1) H2/16) for ALL 8 owned actors (lane = actor x 4 k sub-lanes),
        // so the head weights are read from shared memory once per step instead of once per actor (the 2 x 8 KB per actor
        // were 1 K cycles of the shared-memory pipe); the 16 slice sums meet in the (idle) Part buffer.
        {
            const int ks = H2 >> 4;                           // H2 % 16 == 0 (rf_plan)
            const int a8 = lane >> 2, ksub = lane & 3;
            const float* hrow = Hb2 + a8 * p.ldh2 + warp * ks;
            const float* wbase = Whs + (warp * ks) * ldwh;
            for (int n8 = 0; n8 < A; n8 += 8) {
                float s8[8];
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) s8[jj] = 0.0f;
                const bool second = (n8 + 4 < ldwh);
                for (int k = ksub; k < ks; k += 4) {
                    const float hv = hrow[k];
                    const float* wr = wbase + k * ldwh + n8;
                    const float4 w0 = *reinterpret_cast<const float4*>(wr);
                    s8[0] = fmaf(hv, w0.x, s8[0]); s8[1] = fmaf(hv, w0.y, s8[1]);
                    s8[2] = fmaf(hv, w0.z, s8[2]); s8[3] = fmaf(hv, w0.w, s8[3]);
                    if (second) {
                        const float4 w1 = *reinterpret_cast<const float4*>(wr + 4);
                        s8[4] = fmaf(hv, w1.x, s8[4]); s8[5] = fmaf(hv, w1.y, s8[5]);
                        s8[6] = fmaf(hv, w1.z, s8[6]); s8[7] = fmaf(hv, w1.w, s8[7]);
                    }
                }
                // sum over the 4 k sub-lanes: after two exchange rounds lane ksub holds outputs 2 ksub', 2 ksub' + 1
                const bool u1 = (lane & 2) != 0, u0 = (lane & 1) != 0;
                float t4[4], t2[2];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float recv = __shfl_xor_sync(0xffffffffu, u1 ? s8[i] : s8[i + 4], 2);
                    t4[i] = (u1 ? s8[i + 4] : s8[i]) + recv;
                }
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const float recv = __shfl_xor_sync(0xffffffffu, u0 ? t4[i] : t4[i + 2], 1);
                    t2[i] = (u0 ? t4[i + 2] : t4[i]) + recv;
                }
                const int j0 = n8 + (u1 ? 4 : 0) + (u0 ? 2 : 0);
                float* dst = Part + ((warp * RF_OWN + a8) * ldwh);
                if (j0 < A) dst[j0] = t2[0];
                if (j0 + 1 < A) dst[j0 + 1] = t2[1];
            }
        }
        RF_STAMP(9, 0);
        __syncthreads();
        RF_STAMP(10, 0);
        float rew = 0.0f, dn = 0.0f;
        int slot = SLOT_NONE;
        // ---- owner warps: action, env step, bookkeeping -- same arithmetic, operand order and Philox keys as
        // sample_one() / synth_env_block() of rollout.cu
        if (owner) {
            const int pos = s_pos[own];
            if (lane < A) {
                const int j = lane;
                float pre = 0.0f;
#pragma unroll 4
                for (int w = 0; w < RF_THREADS / 32; ++w) pre += Part[(w * RF_OWN + own) * ldwh + j];    // fixed order
                RF_STAMP(19, 0);
                const float mu = rf_act(pre + Bhs[j], p.act[2]);
                const float sd = Sd[own * A + j];
                float a = mu;
                if (!p.deterministic) a = __fadd_rn(__fmul_rn(Zn[own * A + j], sd), mu);
                a = fminf(fmaxf(a, -1.0f), 1.0f);
                Ac[own * A + j] = a;
                if (valid) {
                    p.stage_act[((long long)i_own * p.n_step + pos) * A + j] = a;
                    p.stage_pd[((long long)i_own * p.n_step + pos) * 2 * A + j] = mu;
                    p.stage_pd[((long long)i_own * p.n_step + pos) * 2 * A + A + j] = sd;
                    if (final_step) {
                        p.action[i_own * A + j] = a;
                        p.pd[i_own * 2 * A + j] = mu;
                        p.pd[i_own * 2 * A + A + j] = sd;
                    }
                }
            }
            __syncwarp();
            RF_STAMP(20, 0);
            float* sown = S + own * D;
            const int ep = s_ep[own] + 1;
            const bool is_done = (p.max_steps > 0) && (ep >= p.max_steps);
            dn = is_done ? 1.0f : 0.0f;
            rew = -Eq[2 * own] / (float)D + 0.1f * Eq[2 * own + 1];
            for (int d = lane; d < D; d += 32) {
                float acc = Eacc[own * D + d];
#pragma unroll 4
                for (int k = 0; k < A; ++k) acc = fmaf(EWa[k * D + d], Ac[own * A + k], acc);
                const float nxt = tanhf(acc) + 0.01f * Egx[own * D + d];
                Nx[own * D + d] = nxt;
                sown[d] = is_done ? Erz[own * D + d] : nxt;
                if (valid && final_step) p.obs_next[i_own * D + d] = nxt;
            }
            RF_STAMP(21, 0);
            if (lane == 0) {
                s_ep[own] = is_done ? 0 : ep;
                if (valid && final_step) {
                    p.reward[i_own] = rew;
                    p.done[i_own] = dn;
                }
                if (valid && pos + 1 == p.n_step) {            // this step completes a window -> next outbox entry
                    const int w = s_cnt[own];
                    if (w < p.Wout) {
                        slot = (int)(i_own * p.Wout + w);
                        p.ev_step[slot] = t;
                        s_cnt[own] = w + 1;
                    } else {
                        slot = SLOT_DROPPED;
                    }
                }
            }
            slot = __shfl_sync(0xffffffffu, slot, 0);
            __syncwarp();
        }
        RF_STAMP(11, 0);
        // ---- window staging (block-wide barriers inside: every warp calls; only owners do work)
        commit_actor(valid, (int)i_own, lane, 32, Nx + own * D, S + own * D, rew, dn, p.n_step, p.stride, D, A, s_pos + own,
                     slot, p.stage_obs, p.stage_act, p.stage_pd, p.stage_rew, p.stage_done, p.o_obs, p.o_act, p.o_pd, p.o_rew,
                     p.o_done);
        RF_STAMP(12, 0);
        // ---- next observation -> z-filter -> every CTA's input tile
        if (owner) {
            const int q4 = lane;                            // D / 4 <= 32 float4 per row
            if (q4 < (D >> 2)) {
                float4 v = *reinterpret_cast<const float4*>(S + own * D + q4 * 4);
                if (i_own >= p.N) v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.zf != nullptr) {
                    const float4 zm = *reinterpret_cast<const float4*>(Zm + q4 * 4);
                    const float4 zs = *reinterpret_cast<const float4*>(Zs + q4 * 4);
                    v.x = fminf(fmaxf((v.x - zm.x) / zs.x, -5.0f), 5.0f);
                    v.y = fminf(fmaxf((v.y - zm.y) / zs.y, -5.0f), 5.0f);
                    v.z = fminf(fmaxf((v.z - zm.z) / zs.z, -5.0f), 5.0f);
                    v.w = fminf(fmaxf((v.w - zm.w) / zs.w, -5.0f), 5.0f);
                    if (i_own >= p.N) v = make_float4(0.f, 0.f, 0.f, 0.f);
                }
                float* qx = X0 + m_own * p.ldx0 + q4 * 4;
                *reinterpret_cast<float4*>(qx) = v;
                const unsigned off = rf_smem_u32(qx) - smem_base;
                if (!final_step) {
#pragma unroll
                    for (int c = 0; c < RF_CS - 1; ++c) rf_st_async_v4(peer_base[c] + off, v, peer_base[c] + bar_off_x0);
                }
            }
        }
        RF_STAMP(13, 0);
    }
    cluster.sync();                                           // nobody leaves while a peer may still address its shared memory

    // ---- write the per-actor control state back
    if (valid) {
        for (int d = lane; d < D; d += 32) p.state[i_own * D + d] = S[own * D + d];
        if (lane == 0) {
            p.stage_pos[i_own] = s_pos[own];
            p.ep_step[i_own] = s_ep[own];
            p.ev_count[i_own] = s_cnt[own];
        }
    }
}

// ---- post-pass 1 (one block): rank the chunk's window completions in (step, actor) order, give them FIFO slots
// with drop-oldest at capacity (fifo_replay.py:27), advance the queue and the shared step counter.
__global__ void __launch_bounds__(1024) ppo_rollout_rank_kernel(const int* __restrict__ ev_step,
                                                                const int* __restrict__ ev_count, int N, int W, int T,
                                                                int* __restrict__ bitmap, int* __restrict__ base,
                                                                int* __restrict__ ev_slot, FifoState* fifo,
                                                                unsigned long long* step_ctr) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int words = (N + 31) >> 5;
    __shared__ int s_total;
    for (int x = tid; x < T * words; x += nt) bitmap[x] = 0;
    for (int x = tid; x <= T; x += nt) base[x] = 0;
    __syncthreads();
    for (int e = tid; e < N * W; e += nt) {
        const int i = e / W, w = e - i * W;
        if (w < ev_count[i]) {
            const int t = ev_step[e];
            atomicOr(&bitmap[t * words + (i >> 5)], 1 << (i & 31));
            atomicAdd(&base[t + 1], 1);
        }
    }
    __syncthreads();
    if (tid == 0) {                                   // T is a few hundred at most: a serial prefix is negligible
        int run = 0;
        for (int t = 0; t <= T; ++t) {
            run += base[t];
            base[t] = run;
        }
        s_total = run;
    }
    __syncthreads();
    const int K = s_total;
    const int cap = fifo->capacity, head = fifo->head, count = fifo->count;
    for (int e = tid; e < N * W; e += nt) {
        const int i = e / W, w = e - i * W;
        int out = SLOT_NONE;
        if (w < ev_count[i]) {
            const int t = ev_step[e];
            int r = base[t];
            const int* bm = bitmap + t * words;
            for (int x = 0; x < (i >> 5); ++x) r += __popc(bm[x]);
            r += __popc(bm[i >> 5] & ((1u << (i & 31)) - 1u));
            out = (K > cap && r < K - cap) ? SLOT_DROPPED : (int)(((long long)head + count + r) % cap);
        }
        ev_slot[e] = out;
    }
    __syncthreads();
    if (tid == 0) {
        int nc = count + K, nh = head, dr = 0;
        if (nc > cap) {
            dr = nc - cap;
            nh = (int)(((long long)head + dr) % cap);
            nc = cap;
        }
        fifo->head = nh;
        fifo->count = nc;
        fifo->dropped += dr;
        fifo->total_in += K;
        if (step_ctr != nullptr) *step_ctr += (unsigned long long)T;
    }
}

// ---- post-pass 2: one block per outbox entry, pure copy into the replay ring
__global__ void __launch_bounds__(256) ppo_rollout_copy_kernel(const int* __restrict__ ev_slot, int n_step, int D, int A,
                                                               const float* __restrict__ o_obs,
                                                               const float* __restrict__ o_act,
                                                               const float* __restrict__ o_pd,
                                                               const float* __restrict__ o_rew,
                                                               const float* __restrict__ o_done,
                                                               float* __restrict__ r_obs, float* __restrict__ r_act,
                                                               float* __restrict__ r_pd, float* __restrict__ r_rew,
                                                               float* __restrict__ r_done) {
    const long long e = blockIdx.x;
    const int slot = ev_slot[e];
    if (slot < 0) return;
    const int g = threadIdx.x, G = blockDim.x;
    copy_floats(r_obs + (long long)slot * (n_step + 1) * D, o_obs + e * (n_step + 1) * D, (n_step + 1) * D, g, G);
    copy_floats(r_act + (long long)slot * n_step * A, o_act + e * n_step * A, n_step * A, g, G);
    copy_floats(r_pd + (long long)slot * n_step * 2 * A, o_pd + e * n_step * 2 * A, n_step * 2 * A, g, G);
    copy_floats(r_rew + (long long)slot * n_step, o_rew + e * n_step, n_step, g, G);
    copy_floats(r_done + (long long)slot * n_step, o_done + e * n_step, n_step, g, G);
}

bool rf_plan(const sb200_mlp* net, int D, int A, RfParams* p, size_t* smem_bytes) {
    if (net == nullptr || net->n_layers != 3 || net->aux_layer >= 0) return false;
    const int H1 = net->dims[1], H2 = net->dims[2];
    if (net->dims[0] != D || net->dims[3] != A) return false;
    if (D % 4 != 0 || D > 128 || A < 1 || A > 32 || H1 % 16 != 0 || H2 % 16 != 0) return false;
    const int Nc1 = H1 / RF_CS, Nc2 = H2 / RF_CS, ldwh = net->ldw[2];
    long long off = 0;
    auto take = [&](long long n) { const long long o = off; off += (n + 3) / 4 * 4; return (int)o; };
    const int oW1 = take((long long)D * Nc1), oW2 = take((long long)H1 * Nc2), oWh = take((long long)H2 * ldwh);
    const int oB = take(Nc1 + Nc2 + ldwh);
    const int ldx0 = D + 4, ldh1 = H1 + 4, ldh2 = H2 + 4;
    const int oX0 = take(RF_ROWS * ldx0), oH1 = take(RF_ROWS * ldh1), oH2 = take(RF_OWN * ldh2);
    // k-split partial tiles of a hidden layer [4][32][max(Nc1, Nc2)] | the head's slice sums [16 warps][8][ldwh]
    const int oPart = take(std::max(4LL * RF_ROWS * std::max(Nc1, Nc2), (long long)(RF_THREADS / 32) * RF_OWN * ldwh));
    const int oZf = take(2 * D), oEnv = take((long long)D * D + A * D);
    const int oS = take(RF_OWN * D), oNext = take(RF_OWN * D), oAct = take(3 * RF_OWN * A);
    const int oPre = take(3 * RF_OWN * D + 2 * RF_OWN);
    if ((size_t)off * sizeof(float) > 224 * 1024) return false;
    // each per-step hand-off counts the bytes a CTA receives from its 3 peers on one mbarrier, whose transaction count
    // must stay below 2^20: hidden layer 1 (32 rows x Nc1), last hidden layer (8 rows x Nc2), next input tile (8 rows x D)
    if (3LL * 4 * std::max({RF_ROWS * Nc1, RF_OWN * Nc2, RF_OWN * D}) >= (1 << 20)) return false;
    if (p != nullptr) {
        p->oW1 = oW1; p->oW2 = oW2; p->oWh = oWh; p->oB = oB; p->oX0 = oX0; p->oH1 = oH1; p->oH2 = oH2; p->oPart = oPart;
        p->oZf = oZf; p->oEnv = oEnv; p->oS = oS; p->oNext = oNext; p->oAct = oAct; p->oPre = oPre;
        p->ldx0 = ldx0; p->ldh1 = ldh1; p->ldh2 = ldh2;
        p->D = D; p->H1 = H1; p->H2 = H2; p->A = A;
    }
    if (smem_bytes != nullptr) *smem_bytes = (size_t)off * sizeof(float);
    return true;
}

}  // namespace

int sb200_rollout_fused_init() {
    SB200_CUDA(cudaFuncSetAttribute(ppo_rollout2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
    return SB200_OK;
}

#ifdef RF_TRACE
extern "C" int sb200_debug_rf_trace(long long* host_out) {
    SB200_CUDA(cudaDeviceSynchronize());
    SB200_CUDA(cudaMemcpyFromSymbol(host_out, g_rf_trace, sizeof(g_rf_trace)));
    return SB200_OK;
}
#endif

extern "C" int sb200_ppo_rollout_supported(const sb200_mlp* net, int D, int A) {
    return rf_plan(net, D, A, nullptr, nullptr) ? 1 : 0;
}

extern "C" size_t sb200_ppo_rollout_scratch_ints(int N, int W, int T) {
    // bitmap [T][ceil(N/32)] | base [T+1] | ev_slot [N*W]
    return (size_t)T * ((N + 31) / 32) + (size_t)(T + 1) + (size_t)N * W;
}

extern "C" int sb200_ppo_rollout_f32(const sb200_ppo_rollout* a, void* stream) {
    SB200_REQUIRE(a != nullptr && a->net != nullptr);
    RfParams p;
    size_t smem = 0;
    if (!rf_plan(a->net, a->D, a->A, &p, &smem)) return SB200_ERR_UNSUPPORTED;
    SB200_REQUIRE(a->N >= 1 && a->T >= 1 && a->n_step >= 1 && a->stride >= 1 && a->W >= 1);
    SB200_REQUIRE(a->state && a->WsT && a->WaT && a->ep_step && a->action && a->pd && a->obs_next && a->reward && a->done);
    SB200_REQUIRE(a->log_var && a->stage_pos && a->stage_obs && a->stage_act && a->stage_pd && a->stage_rew && a->stage_done);
    SB200_REQUIRE(a->o_obs && a->o_act && a->o_pd && a->o_rew && a->o_done && a->ev_step && a->ev_count);
    for (int l = 0; l < 3; ++l) {
        p.W[l] = a->net->W[l];
        p.b[l] = a->net->b[l];
        p.ldw[l] = a->net->ldw[l];
        p.act[l] = a->net->act[l];
        SB200_REQUIRE(p.W[l] != nullptr && p.b[l] != nullptr && p.ldw[l] % 4 == 0 && (((uintptr_t)p.W[l]) & 15) == 0);
    }
    SB200_REQUIRE((((uintptr_t)a->WsT) & 15) == 0 && (((uintptr_t)a->WaT) & 15) == 0 && (((uintptr_t)a->state) & 15) == 0);
    p.zf = a->zf_stats;
    p.zf_eps = a->zf_eps;
    p.log_var = a->log_var;
    p.log_noise = a->log_noise;
    p.agent_seed = a->agent_seed;
    p.deterministic = a->deterministic;
    p.state = a->state;
    p.WsT = a->WsT;
    p.WaT = a->WaT;
    p.ep_step = a->ep_step;
    p.max_steps = a->max_steps;
    p.env_seed = a->env_seed;
    p.action = a->action;
    p.pd = a->pd;
    p.obs_next = a->obs_next;
    p.reward = a->reward;
    p.done = a->done;
    p.stage_pos = a->stage_pos;
    p.stage_obs = a->stage_obs;
    p.stage_act = a->stage_act;
    p.stage_pd = a->stage_pd;
    p.stage_rew = a->stage_rew;
    p.stage_done = a->stage_done;
    p.o_obs = a->o_obs;
    p.o_act = a->o_act;
    p.o_pd = a->o_pd;
    p.o_rew = a->o_rew;
    p.o_done = a->o_done;
    p.ev_step = a->ev_step;
    p.ev_count = a->ev_count;
    p.Wout = a->W;
    p.N = a->N;
    p.n_step = a->n_step;
    p.stride = a->stride;
    p.T = a->T;
    p.step_ctr = (const unsigned long long*)a->step_counter;
    const long long clusters = ((long long)a->N + RF_ROWS - 1) / RF_ROWS;
    ppo_rollout2_kernel<<<(unsigned)(clusters * RF_CS), RF_THREADS, smem, (cudaStream_t)stream>>>(p);
    return sb200_launch_status();
}

extern "C" int sb200_ppo_rollout_commit_f32(const sb200_ppo_rollout* a, int* scratch, void* fifo_state, float* r_obs,
                                            float* r_act, float* r_pd, float* r_rew, float* r_done,
                                            uint64_t* step_counter, void* stream) {
    SB200_REQUIRE(a != nullptr && scratch != nullptr && fifo_state != nullptr);
    SB200_REQUIRE(r_obs && r_act && r_pd && r_rew && r_done && step_counter);
    SB200_REQUIRE(a->N >= 1 && a->T >= 1 && a->W >= 1 && a->ev_step && a->ev_count);
    const int words = (a->N + 31) / 32;
    int* bitmap = scratch;
    int* base = bitmap + (size_t)a->T * words;
    int* ev_slot = base + (a->T + 1);
    cudaStream_t st = (cudaStream_t)stream;
    ppo_rollout_rank_kernel<<<1, 1024, 0, st>>>(a->ev_step, a->ev_count, a->N, a->W, a->T, bitmap, base, ev_slot,
                                                (FifoState*)fifo_state, (unsigned long long*)step_counter);
    ppo_rollout_copy_kernel<<<(unsigned)((long long)a->N * a->W), 256, 0, st>>>(
        ev_slot, a->n_step, a->D, a->A, a->o_obs, a->o_act, a->o_pd, a->o_rew, a->o_done, r_obs, r_act, r_pd, r_rew,
        r_done);
    return sb200_launch_status(2);
}
