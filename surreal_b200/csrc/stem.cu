// CNN stem of the pixel path (surreal/model/model_builders/builders.py:8-33, ppo_net.py:268-273,368-375):
//   uint8 frames / 255 -> Conv2d(16, k8, s4) + ReLU -> Conv2d(32, k4, s2) + ReLU -> Flatten -> Linear(cnn_feature_dim) + ReLU
// (VALID padding; the Linear layer runs on the MLP kernels / the tcgen05 linear kernel).  This file holds the two
// convolutions, forward and backward, as direct fp32 FFMA kernels:
//
//   conv_fwd_kernel   one frame per CTA iteration, the frame (converted to float, x 1/255 for uint8 input) and the layer's
//                     weights live in shared memory; a thread owns 4 consecutive output columns x 4 output channels and
//                     walks the taps with the input row segment in registers (13 LDS.128 per 128 FMA for k8 s4).
//   conv_bwd_dw_kernel  weight / bias gradient: a thread owns one tap (c, ky, kx) x all output channels, frames are spread
//                     over CTAs which write PARTIAL gradients into slabs (reduced in a fixed order by
//                     sb200_grad_reduce_norm_f32, like the MLP layers: deterministic, no atomics).
//   conv_bwd_dx_kernel  input gradient of the second convolution (times relu' of the first one's output).
//
// Layouts: frames [rows][C][H][W] (torch NCHW, uint8 or float); conv output [rows][COUT][HO][WO] so that Flatten matches
// torch's (c, h, w) order; conv weights in the KERNEL layout Wk[(c*KS + ky)*KS + kx][COUT] (transpose of torch's
// [COUT][C][KS][KS]), bias [COUT].  Frames stay uint8 in HBM: 28 224 B per 4x84x84 frame (SURVEY §8d).
#include "common.cuh"

namespace {

constexpr int CT = 256;

template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<unsigned char>(unsigned char v) { return (float)v; }

__host__ __device__ inline int ru4(int v) { return (v + 3) & ~3; }

// shared-memory pitch of one input row: enough columns for the last (partly masked) group of 4 outputs
template <int KS, int ST> __host__ __device__ inline int row_pitch(int W) { return ru4(W + 3 * ST + KS); }

template <int KS, int ST, int COUT, typename IN_T>
__global__ void __launch_bounds__(CT) conv_fwd_kernel(const IN_T* __restrict__ x, int frames, int CIN, int H, int W,
                                                      const float* __restrict__ Wk, const float* __restrict__ bias,
                                                      float in_scale, float* __restrict__ y, long long fsz) {
    extern __shared__ __align__(16) float sm[];
    const int HO = (H - KS) / ST + 1, WO = (W - KS) / ST + 1;
    const int Wp = row_pitch<KS, ST>(W);
    const int taps = CIN * KS * KS;
    float* ws = sm;                          // [taps][COUT]
    float* xs = sm + taps * COUT;            // [CIN][H][Wp]
    const int tid = threadIdx.x;
    for (int i = tid; i < taps * COUT / 4; i += CT)
        reinterpret_cast<float4*>(ws)[i] = reinterpret_cast<const float4*>(Wk)[i];
    for (int i = tid; i < CIN * H * Wp; i += CT) xs[i] = 0.0f;            // padding columns stay zero
    __syncthreads();
    constexpr int CQ = COUT / 4;
    constexpr int SPAN = 3 * ST + KS;
    const int groups = (WO + 3) / 4;
    const int items = HO * groups * CQ;
    for (int f = blockIdx.x; f < frames; f += gridDim.x) {
        const IN_T* xf = x + (long long)f * fsz;
        for (int i = tid; i < CIN * H * W; i += CT) {
            const int c = i / (H * W), r = i - c * H * W, yy = r / W, xx = r - yy * W;
            xs[(c * H + yy) * Wp + xx] = to_f<IN_T>(xf[i]) * in_scale;
        }
        __syncthreads();
        for (int it = tid; it < items; it += CT) {
            const int cq = it % CQ;
            const int g = (it / CQ) % groups;
            const int oy = it / (CQ * groups);
            const int ox0 = g * 4;
            float acc[4][4];
#pragma unroll
            for (int p = 0; p < 4; ++p)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[p][j] = 0.0f;
            for (int c = 0; c < CIN; ++c) {
#pragma unroll
                for (int ky = 0; ky < KS; ++ky) {
                    const float* xr = xs + (c * H + oy * ST + ky) * Wp + ox0 * ST;
                    float xin[SPAN];
#pragma unroll
                    for (int i = 0; i < SPAN; ++i) xin[i] = xr[i];
                    const float* wr = ws + ((c * KS + ky) * KS) * COUT + cq * 4;
#pragma unroll
                    for (int kx = 0; kx < KS; ++kx) {
                        const float4 w4 = *reinterpret_cast<const float4*>(wr + kx * COUT);
#pragma unroll
                        for (int p = 0; p < 4; ++p) {
                            const float v = xin[p * ST + kx];
                            acc[p][0] = fmaf(v, w4.x, acc[p][0]);
                            acc[p][1] = fmaf(v, w4.y, acc[p][1]);
                            acc[p][2] = fmaf(v, w4.z, acc[p][2]);
                            acc[p][3] = fmaf(v, w4.w, acc[p][3]);
                        }
                    }
                }
            }
            float* yf = y + (long long)f * COUT * HO * WO;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int co = cq * 4 + j;
                const float b = bias[co];
#pragma unroll
                for (int p = 0; p < 4; ++p)
                    if (ox0 + p < WO) yf[(co * HO + oy) * WO + ox0 + p] = fmaxf(acc[p][j] + b, 0.0f);
            }
        }
        __syncthreads();
    }
}

// dW[(c,ky,kx)][co] = sum_{f,oy,ox} dY[f][co][oy][ox] * X[f][c][oy*ST+ky][ox*ST+kx] * in_scale,  db[co] = sum dY.
// CTA b accumulates frames b, b+grid, ... and writes its partial sums into slab b: [taps*COUT | COUT(pad 4)].
template <int KS, int ST, int COUT, typename IN_T>
__global__ void __launch_bounds__(CT) conv_bwd_dw_kernel(const IN_T* __restrict__ x, const float* __restrict__ dy, int frames,
                                                         int CIN, int H, int W, float in_scale, float* __restrict__ slab_w,
                                                         float* __restrict__ slab_b, long long slab_stride, long long fsz) {
    extern __shared__ __align__(16) float sm[];
    const int HO = (H - KS) / ST + 1, WO = (W - KS) / ST + 1;
    const int taps = CIN * KS * KS, npos = HO * WO, npos4 = ru4(npos);
    float* xs = sm;                          // [CIN][H][W]
    float* ds = sm + ru4(CIN * H * W);       // [npos][COUT] (position-major: one LDS.128 broadcast per 4 channels)
    const int tid = threadIdx.x;
    float* out_w = slab_w + (long long)blockIdx.x * slab_stride;
    float* out_b = slab_b + (long long)blockIdx.x * slab_stride;
    (void)npos4;
    for (int t0 = 0; t0 < taps; t0 += CT) {
        const int tap = t0 + tid;
        const bool on = tap < taps;
        const int c = on ? tap / (KS * KS) : 0, r = on ? tap - c * KS * KS : 0, ky = r / KS, kx = r - ky * KS;
        float acc[COUT];
#pragma unroll
        for (int j = 0; j < COUT; ++j) acc[j] = 0.0f;
        float bacc = 0.0f;                    // thread j < COUT also sums dY of channel j (first tap batch only)
        for (int f = blockIdx.x; f < frames; f += gridDim.x) {
            __syncthreads();
            const IN_T* xf = x + (long long)f * fsz;
            for (int i = tid; i < CIN * H * W; i += CT) xs[i] = to_f<IN_T>(xf[i]) * in_scale;
            const float* df = dy + (long long)f * COUT * npos;
            for (int i = tid; i < COUT * npos; i += CT) {
                const int co = i / npos, p = i - co * npos;
                ds[p * COUT + co] = df[i];
            }
            __syncthreads();
            if (on) {
                for (int oy = 0; oy < HO; ++oy) {
                    const float* xr = xs + (c * H + oy * ST + ky) * W + kx;
                    for (int ox = 0; ox < WO; ++ox) {
                        const float v = xr[ox * ST];
                        const float4* d4 = reinterpret_cast<const float4*>(ds + (oy * WO + ox) * COUT);
#pragma unroll
                        for (int j = 0; j < COUT / 4; ++j) {
                            const float4 d = d4[j];
                            acc[4 * j + 0] = fmaf(v, d.x, acc[4 * j + 0]);
                            acc[4 * j + 1] = fmaf(v, d.y, acc[4 * j + 1]);
                            acc[4 * j + 2] = fmaf(v, d.z, acc[4 * j + 2]);
                            acc[4 * j + 3] = fmaf(v, d.w, acc[4 * j + 3]);
                        }
                    }
                }
            }
            if (t0 == 0 && tid < COUT)
                for (int p = 0; p < npos; ++p) bacc += ds[p * COUT + tid];
        }
        if (on) {
#pragma unroll
            for (int j = 0; j < COUT; ++j) out_w[(long long)tap * COUT + j] = acc[j];
        }
        if (t0 == 0 && tid < COUT) out_b[tid] = bacc;
    }
}

// dX[f][c][y][x] = relu'(A[f][c][y][x]) * sum_{co,ky,kx} dY[f][co][(y-ky)/ST][(x-kx)/ST] * Wk[(c,ky,kx)][co]
template <int KS, int ST, int COUT>
__global__ void __launch_bounds__(CT) conv_bwd_dx_kernel(const float* __restrict__ dy, const float* __restrict__ Wk,
                                                         const float* __restrict__ act, int frames, int CIN, int H, int W,
                                                         float* __restrict__ dx) {
    extern __shared__ __align__(16) float sm[];
    const int HO = (H - KS) / ST + 1, WO = (W - KS) / ST + 1;
    const int taps = CIN * KS * KS, npos = HO * WO;
    float* ws = sm;                          // [taps][COUT]
    float* ds = sm + taps * COUT;            // [npos][COUT]
    const int tid = threadIdx.x;
    for (int i = tid; i < taps * COUT / 4; i += CT)
        reinterpret_cast<float4*>(ws)[i] = reinterpret_cast<const float4*>(Wk)[i];
    for (int f = blockIdx.x; f < frames; f += gridDim.x) {
        __syncthreads();
        const float* df = dy + (long long)f * COUT * npos;
        for (int i = tid; i < COUT * npos; i += CT) {
            const int co = i / npos, p = i - co * npos;
            ds[p * COUT + co] = df[i];
        }
        __syncthreads();
        const long long base = (long long)f * CIN * H * W;
        for (int i = tid; i < CIN * H * W; i += CT) {
            const int c = i / (H * W), r = i - c * H * W, yy = r / W, xx = r - yy * W;
            float s = 0.0f;
            if (act == nullptr || act[base + i] > 0.0f) {
                for (int ky = yy % ST; ky < KS; ky += ST) {
                    const int oy = (yy - ky) / ST;
                    if (yy - ky < 0 || oy >= HO) continue;
                    for (int kx = xx % ST; kx < KS; kx += ST) {
                        const int ox = (xx - kx) / ST;
                        if (xx - kx < 0 || ox >= WO) continue;
                        const float4* d4 = reinterpret_cast<const float4*>(ds + (oy * WO + ox) * COUT);
                        const float4* w4 = reinterpret_cast<const float4*>(ws + ((c * KS + ky) * KS + kx) * COUT);
#pragma unroll
                        for (int j = 0; j < COUT / 4; ++j) {
                            const float4 d = d4[j], w = w4[j];
                            s = fmaf(d.x, w.x, s); s = fmaf(d.y, w.y, s); s = fmaf(d.z, w.z, s); s = fmaf(d.w, w.w, s);
                        }
                    }
                }
            }
            dx[base + i] = s;
        }
    }
}

constexpr size_t STEM_SMEM_MAX = 200 * 1024;

template <int KS, int ST, int COUT, typename IN_T>
int launch_fwd(const void* x, int frames, int CIN, int H, int W, const float* Wk, const float* bias, float in_scale, float* y,
               cudaStream_t st, long long fsz) {
    const size_t smem = ((size_t)CIN * KS * KS * COUT + (size_t)CIN * H * row_pitch<KS, ST>(W)) * sizeof(float);
    if (smem > STEM_SMEM_MAX) return SB200_ERR_UNSUPPORTED;
    const int grid = frames < 148 * 4 ? frames : 148 * 4;
    conv_fwd_kernel<KS, ST, COUT, IN_T><<<grid, CT, smem, st>>>((const IN_T*)x, frames, CIN, H, W, Wk, bias, in_scale, y, fsz);
    return sb200_launch_status();
}

template <int KS, int ST, int COUT, typename IN_T>
int launch_dw(const void* x, const float* dy, int frames, int CIN, int H, int W, float in_scale, float* slab_w, float* slab_b,
              long long slab_stride, int splits, cudaStream_t st, long long fsz) {
    const int HO = (H - KS) / ST + 1, WO = (W - KS) / ST + 1;
    const size_t smem = ((size_t)ru4(CIN * H * W) + (size_t)HO * WO * COUT) * sizeof(float);
    if (smem > STEM_SMEM_MAX) return SB200_ERR_UNSUPPORTED;
    conv_bwd_dw_kernel<KS, ST, COUT, IN_T><<<splits, CT, smem, st>>>((const IN_T*)x, dy, frames, CIN, H, W, in_scale, slab_w, slab_b,
                                                                     slab_stride, fsz);
    return sb200_launch_status();
}

}  // namespace

// called once from sb200_init(): every instantiation may use the large dynamic shared-memory carve-out
int sb200_stem_init() {
    const int m = (int)STEM_SMEM_MAX;
    SB200_CUDA(cudaFuncSetAttribute(conv_fwd_kernel<8, 4, 16, unsigned char>, cudaFuncAttributeMaxDynamicSharedMemorySize, m));
    SB200_CUDA(cudaFuncSetAttribute(conv_fwd_kernel<8, 4, 16, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, m));
    SB200_CUDA(cudaFuncSetAttribute(conv_fwd_kernel<4, 2, 32, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, m));
    SB200_CUDA(cudaFuncSetAttribute(conv_bwd_dw_kernel<8, 4, 16, unsigned char>, cudaFuncAttributeMaxDynamicSharedMemorySize, m));
    SB200_CUDA(cudaFuncSetAttribute(conv_bwd_dw_kernel<8, 4, 16, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, m));
    SB200_CUDA(cudaFuncSetAttribute(conv_bwd_dw_kernel<4, 2, 32, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, m));
    SB200_CUDA(cudaFuncSetAttribute(conv_bwd_dx_kernel<4, 2, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, m));
    return SB200_OK;
}

// layer: 1 = Conv2d(16, k8, s4), 2 = Conv2d(32, k4, s2) (CNNStemNetwork's fixed architecture, builders.py:9).
// in_u8: input frames are uint8 (scaled by in_scale = 1/255, ppo_net.py:370) instead of float.
extern "C" int sb200_conv_forward_f32(int layer, const void* x, int in_u8, int64_t frames, int CIN, int H, int W, const float* Wk,
                                      const float* bias, double in_scale, float* y, void* stream) {
    SB200_REQUIRE(x && Wk && bias && y && frames >= 0 && CIN >= 1 && (layer == 1 || layer == 2));
    SB200_REQUIRE((((uintptr_t)Wk) & 15) == 0);
    if (layer == 1 && in_u8) return sb200_conv1_forward_u8_strided(x, (int64_t)CIN * H * W, frames, CIN, H, W, Wk, bias, in_scale, y,
                                                                   stream);
    if (frames == 0) return SB200_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const long long fsz = (long long)CIN * H * W;
    if (layer == 1) {
        SB200_REQUIRE(H >= 8 && W >= 8);
        return launch_fwd<8, 4, 16, float>(x, (int)frames, CIN, H, W, Wk, bias, (float)in_scale, y, st, fsz);
    }
    SB200_REQUIRE(H >= 4 && W >= 4 && !in_u8);
    return launch_fwd<4, 2, 32, float>(x, (int)frames, CIN, H, W, Wk, bias, (float)in_scale, y, st, fsz);
}

// Conv layer 1 on uint8 frames that sit `row_bytes` apart (>= CIN*H*W): frames read in place from wider records, e.g. the
// mixed pixel + low-dim observation rows of the staging / replay buffers (utils.obs_layout).
extern "C" int sb200_conv1_forward_u8_strided(const void* x, int64_t row_bytes, int64_t frames, int CIN, int H, int W,
                                              const float* Wk, const float* bias, double in_scale, float* y, void* stream) {
    SB200_REQUIRE(x && Wk && bias && y && frames >= 0 && CIN >= 1);
    SB200_REQUIRE((((uintptr_t)Wk) & 15) == 0 && row_bytes >= (int64_t)CIN * H * W);
    if (frames == 0) return SB200_OK;
    SB200_REQUIRE(H >= 8 && W >= 8);
    return launch_fwd<8, 4, 16, unsigned char>(x, (int)frames, CIN, H, W, Wk, bias, (float)in_scale, y, (cudaStream_t)stream,
                                               (long long)row_bytes);
}

// Partial weight / bias gradients of `frames` frames into `splits` slabs (slab s at slab_w + s*slab_stride, bias part at
// slab_b + s*slab_stride); dy is the gradient w.r.t. the layer's PRE-activation output [frames][COUT][HO][WO].
extern "C" int sb200_conv_backward_dw_f32(int layer, const void* x, int in_u8, const float* dy, int64_t frames, int CIN, int H,
                                          int W, double in_scale, float* slab_w, float* slab_b, int64_t slab_stride, int splits,
                                          void* stream) {
    SB200_REQUIRE(x && dy && slab_w && slab_b && frames >= 1 && CIN >= 1 && splits >= 1 && (layer == 1 || layer == 2));
    if (layer == 1 && in_u8)
        return sb200_conv1_backward_dw_u8_strided(x, (int64_t)CIN * H * W, dy, frames, CIN, H, W, in_scale, slab_w, slab_b,
                                                  slab_stride, splits, stream);
    cudaStream_t st = (cudaStream_t)stream;
    const long long fsz = (long long)CIN * H * W;
    if (layer == 1)
        return launch_dw<8, 4, 16, float>(x, dy, (int)frames, CIN, H, W, (float)in_scale, slab_w, slab_b, slab_stride, splits, st, fsz);
    SB200_REQUIRE(!in_u8);
    return launch_dw<4, 2, 32, float>(x, dy, (int)frames, CIN, H, W, (float)in_scale, slab_w, slab_b, slab_stride, splits, st, fsz);
}

// sb200_conv_backward_dw_f32 of layer 1 on uint8 frames `row_bytes` apart (see sb200_conv1_forward_u8_strided).
extern "C" int sb200_conv1_backward_dw_u8_strided(const void* x, int64_t row_bytes, const float* dy, int64_t frames, int CIN,
                                                  int H, int W, double in_scale, float* slab_w, float* slab_b, int64_t slab_stride,
                                                  int splits, void* stream) {
    SB200_REQUIRE(x && dy && slab_w && slab_b && frames >= 1 && CIN >= 1 && splits >= 1);
    SB200_REQUIRE(row_bytes >= (int64_t)CIN * H * W);
    return launch_dw<8, 4, 16, unsigned char>(x, dy, (int)frames, CIN, H, W, (float)in_scale, slab_w, slab_b, slab_stride, splits,
                                              (cudaStream_t)stream, (long long)row_bytes);
}

// dx[frames][CIN][H][W] = relu'(act) * conv_transpose(dy, Wk) for layer 2 (its input is layer 1's post-ReLU output `act`).
extern "C" int sb200_conv_backward_dx_f32(int layer, const float* dy, const float* Wk, const float* act, int64_t frames, int CIN,
                                          int H, int W, float* dx, void* stream) {
    SB200_REQUIRE(dy && Wk && dx && frames >= 1 && layer == 2 && CIN >= 1);
    const int HO = (H - 4) / 2 + 1, WO = (W - 4) / 2 + 1;
    const size_t smem = ((size_t)CIN * 16 * 32 + (size_t)HO * WO * 32) * sizeof(float);
    if (smem > STEM_SMEM_MAX) return SB200_ERR_UNSUPPORTED;
    const int grid = frames < 148 * 4 ? (int)frames : 148 * 4;
    conv_bwd_dx_kernel<4, 2, 32><<<grid, CT, smem, (cudaStream_t)stream>>>(dy, Wk, act, (int)frames, CIN, H, W, dx);
    return sb200_launch_status();
}

// ------------------------------------------------------------------------------------------------------------------------
// Synthetic PIXEL environment of BASELINE configs[3] (SURVEY §8d cfg 4): every step each actor observes a fresh frame of
// uniform random bytes (Philox keyed by (seed, step, actor, word)), reward = -mean(a^2) + 0.1 xi, done at the episode cap.
// Frames are written as 32-bit words (4 pixels each); `state` = what the actor observes next (a reset frame where done),
// `obs_next` = the true successor.
namespace {
__global__ void __launch_bounds__(256) synth_pixel_env_kernel(unsigned int* __restrict__ state, const float* __restrict__ action, int N,
                                                              int words, int A, int max_steps, int* __restrict__ ep_step,
                                                              unsigned long long seed, const unsigned long long* __restrict__ step_ctr,
                                                              unsigned int* __restrict__ obs_next, float* __restrict__ reward,
                                                              float* __restrict__ done) {
    const int i = blockIdx.y;
    const unsigned long long ctr = (step_ctr != nullptr) ? *step_ctr : 0ull;
    const int t = ep_step[i] + 1;
    const bool dn = (max_steps > 0) && (t >= max_steps);
    const int w4 = words / 4;
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < w4; g += gridDim.x * blockDim.x) {
        const Philox4 r = philox4x32_10(seed ^ 0x2545F4914F6CDD1Dull, ctr, ((unsigned long long)i << 24) | (unsigned long long)g);
        uint4 nx = make_uint4(r.x, r.y, r.z, r.w);
        reinterpret_cast<uint4*>(obs_next + (long long)i * words)[g] = nx;
        if (dn) {
            const Philox4 z = philox4x32_10(seed ^ 0x9E3779B97F4A7C15ull, ctr, ((unsigned long long)i << 24) | (unsigned long long)g);
            nx = make_uint4(z.x, z.y, z.z, z.w);
        }
        reinterpret_cast<uint4*>(state + (long long)i * words)[g] = nx;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        float s = 0.0f;
        for (int j = 0; j < A; ++j) s += action[(long long)i * A + j] * action[(long long)i * A + j];
        const Philox4 r = philox4x32_10(seed ^ 0x5851F42D4C957F2Dull, ctr, ((unsigned long long)i << 24) | 0xFFFFFFull);
        reward[i] = -s / (float)A + 0.1f * box_muller(r.x, r.y).x;
        done[i] = dn ? 1.0f : 0.0f;
    }
}
// ep_step update must happen after every block has read it: separate tiny kernel
__global__ void synth_pixel_env_tick_kernel(int N, int max_steps, int* __restrict__ ep_step) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int t = ep_step[i] + 1;
    ep_step[i] = ((max_steps > 0) && (t >= max_steps)) ? 0 : t;
}
}  // namespace

extern "C" int sb200_synth_pixel_env_step_u8(void* state, const float* action, int N, int64_t frame_bytes, int A, int max_steps,
                                             int* ep_step, uint64_t seed, const uint64_t* step_counter, void* obs_next,
                                             float* reward, float* done, void* stream) {
    SB200_REQUIRE(state && action && ep_step && obs_next && reward && done && N >= 1 && A >= 1);
    SB200_REQUIRE(frame_bytes >= 16 && frame_bytes % 16 == 0 && frame_bytes / 16 < (1ll << 24) && N < (1 << 24));
    const int words = (int)(frame_bytes / 4);
    dim3 grid((unsigned)((words / 4 + 255) / 256 < 8 ? (words / 4 + 255) / 256 : 8), (unsigned)N);
    synth_pixel_env_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((unsigned int*)state, action, N, words, A, max_steps, ep_step,
                                                                   (unsigned long long)seed, (const unsigned long long*)step_counter,
                                                                   (unsigned int*)obs_next, reward, done);
    synth_pixel_env_tick_kernel<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(N, max_steps, ep_step);
    return sb200_launch_status(2);
}

// ------------------------------------------------------------------------------------------------------------------------
// Synthetic MIXED environment: one camera frame plus a low-dim state per actor, written straight into the packed observation
// rows the staging / replay kernels copy as opaque words (utils.obs_layout): row = [frame as frame_words 32-bit words |
// D low-dim floats | zero padding to row_words].  The frame part is SyntheticPixelEnv's (same Philox keys: the same bytes for
// the same seed and step), the low-dim part, the reward and done are SyntheticEnv's (s' = tanh(Ws s + Wa a) + 0.01 xi,
// r = -|s|^2 / D + 0.1 xi', same keys and FMA order).  One CTA per actor, so the episode counter is updated in-kernel.
namespace {
__global__ void __launch_bounds__(256) synth_mixed_env_kernel(float* __restrict__ state, const float* __restrict__ action,
                                                              const float* __restrict__ Ws, const float* __restrict__ Wa, int D,
                                                              int A, int frame_words, long long row_words, int max_steps,
                                                              int* __restrict__ ep_step, unsigned long long seed,
                                                              const unsigned long long* __restrict__ step_ctr,
                                                              float* __restrict__ obs_next, float* __restrict__ reward,
                                                              float* __restrict__ done) {
    extern __shared__ float sm[];            // [D] low-dim state, [A] action
    __shared__ float s_q;
    float* s_s = sm;
    float* s_a = sm + D;
    const int i = blockIdx.x, tid = threadIdx.x;
    float* row = state + (long long)i * row_words;
    float* nrow = obs_next + (long long)i * row_words;
    for (int d = tid; d < D; d += 256) s_s[d] = row[frame_words + d];
    for (int j = tid; j < A; j += 256) s_a[j] = action[(long long)i * A + j];
    const unsigned long long ctr = (step_ctr != nullptr) ? *step_ctr : 0ull;
    const int t = ep_step[i] + 1;
    const bool dn = (max_steps > 0) && (t >= max_steps);
    __syncthreads();
    // frame: 4 words (16 pixels) per Philox draw
    uint4* fr = reinterpret_cast<uint4*>(row);
    uint4* nfr = reinterpret_cast<uint4*>(nrow);
    for (int g = tid; g < frame_words / 4; g += 256) {
        const Philox4 r = philox4x32_10(seed ^ 0x2545F4914F6CDD1Dull, ctr, ((unsigned long long)i << 24) | (unsigned long long)g);
        uint4 nx = make_uint4(r.x, r.y, r.z, r.w);
        nfr[g] = nx;
        if (dn) {
            const Philox4 z = philox4x32_10(seed ^ 0x9E3779B97F4A7C15ull, ctr, ((unsigned long long)i << 24) | (unsigned long long)g);
            nx = make_uint4(z.x, z.y, z.z, z.w);
        }
        fr[g] = nx;
    }
    if (tid < 32) {
        float q = 0.0f;
        for (int d = tid; d < D; d += 32) q += s_s[d] * s_s[d];
        q = warp_sum(q);
        if (tid == 0) s_q = q;
    }
    __syncthreads();
    for (int d = tid; d < D; d += 256) {
        float acc = 0.0f;
#pragma unroll 8
        for (int k = 0; k < D; ++k) acc = fmaf(__ldg(Ws + (long long)k * D + d), s_s[k], acc);
#pragma unroll 4
        for (int k = 0; k < A; ++k) acc = fmaf(__ldg(Wa + (long long)k * D + d), s_a[k], acc);
        const Philox4 r = philox4x32_10(seed ^ 0x5851F42D4C957F2Dull, ctr, ((unsigned long long)i << 20) | (unsigned long long)d);
        const float2 g = box_muller(r.x, r.y);
        const float nxt = tanhf(acc) + 0.01f * g.x;
        nrow[frame_words + d] = nxt;
        row[frame_words + d] = dn ? box_muller(r.z, r.w).x : nxt;
        if (d == 0) {
            reward[i] = -s_q / (float)D + 0.1f * g.y;
            done[i] = dn ? 1.0f : 0.0f;
        }
    }
    __syncthreads();                         // every thread has read ep_step[i]
    if (tid == 0) ep_step[i] = dn ? 0 : t;
}
}  // namespace

extern "C" int sb200_synth_mixed_env_step_f32(float* state, const float* action, const float* Ws, const float* Wa, int N, int D,
                                              int A, int frame_words, int64_t row_words, int max_steps, int* ep_step, uint64_t seed,
                                              const uint64_t* step_counter, float* obs_next, float* reward, float* done,
                                              void* stream) {
    SB200_REQUIRE(state && action && Ws && Wa && ep_step && obs_next && reward && done && N >= 1 && D >= 1 && A >= 1);
    SB200_REQUIRE(frame_words >= 4 && frame_words % 4 == 0 && frame_words / 4 < (1 << 24) && D < (1 << 20));
    SB200_REQUIRE(row_words >= (int64_t)frame_words + D && row_words % 4 == 0);
    SB200_REQUIRE((((uintptr_t)state) & 15) == 0 && (((uintptr_t)obs_next) & 15) == 0);
    SB200_REQUIRE((size_t)(D + A) * sizeof(float) <= 40 * 1024);
    synth_mixed_env_kernel<<<N, 256, (size_t)(D + A) * sizeof(float), (cudaStream_t)stream>>>(
        state, action, Ws, Wa, D, A, frame_words, (long long)row_words, max_steps, ep_step, (unsigned long long)seed,
        (const unsigned long long*)step_counter, obs_next, reward, done);
    return sb200_launch_status();
}
