// net_fp32.cu -- DualNetwork forward pieces on CUDA cores:
//   * conv_input (3->128, K = 27: too thin for the tensor pipe) + folded BN + ReLU
//   * the fp32 "parity numerics" trunk (16 residual blocks as direct 3x3 convolutions)
//   * the policy / value heads (1x1 convs, FCs, softmax, tanh), shared by both trunks
//
// Replaces DualNetwork.forward (dual_network.py:89-121) as called from pv_mcts_cpp.py:61-69.
// BatchNorm is eval-mode (running statistics, eps 1e-5) and folded at upload time:
// scale into the conv weights, shift as a per-channel bias.
// Spatial index = picture cell R*9+C (the (3,9,9) planes of cpp/uttt_game.cpp:244-280 after the
// NHWC->NCHW transpose); channel is the fastest-varying dimension of every activation buffer.
#include "common.cuh"
#include "heads_fc.cuh"

namespace uttt {

// ---------------------------------------------------------------- conv_input (dual_network.py:93-95)
// planes: bf16 [row][3][81]; out: fp32 [row][81][128].  One block per position, thread = channel.
__global__ void __launch_bounds__(128) conv_input_kernel(const __nv_bfloat16* __restrict__ planes,
                                                         const float* __restrict__ w /*[9][3][128]*/,
                                                         const float* __restrict__ b, const int32_t* __restrict__ count,
                                                         float* __restrict__ out) {
    int row = blockIdx.x;
    if (row >= *count) return;
    __shared__ float in[3][11][11];
    for (int i = threadIdx.x; i < 3 * 121; i += 128) (&in[0][0][0])[i] = 0.0f;
    __syncthreads();
    for (int i = threadIdx.x; i < 243; i += 128) {
        int ch = i / 81, cell = i - 81 * ch;
        in[ch][cell / 9 + 1][cell % 9 + 1] = __bfloat162float(planes[(size_t)row * 243 + i]);
    }
    __syncthreads();
    int co = threadIdx.x;
    float wr[27];
#pragma unroll
    for (int i = 0; i < 27; i++) wr[i] = w[i * 128 + co];
    float bias = b[co];
    for (int cell = 0; cell < 81; cell++) {
        int r = cell / 9, c = cell - 9 * r;
        float acc = bias;
#pragma unroll
        for (int tap = 0; tap < 9; tap++)
#pragma unroll
            for (int ci = 0; ci < 3; ci++) acc = fmaf(in[ci][r + tap / 3][c + tap % 3], wr[tap * 3 + ci], acc);
        out[((size_t)row * 81 + cell) * 128 + co] = fmaxf(acc, 0.0f);
    }
}

// ---------------------------------------------------------------- fp32 3x3 conv layer
// in/out: [row][81][128] fp32; w: [9][128 cin][128 cout] (BN scale folded); epilogue: +bias (+resid) ReLU.
// One block (256 threads) per position; input staged in shared memory with a zero halo (11x11x128).
// lane -> 4 consecutive output channels, warp -> cells {warp, warp+8, ...}.
constexpr int F32_THREADS = 256;
constexpr int F32_SMEM = 121 * 128 * 4;

__global__ void __launch_bounds__(F32_THREADS) conv3x3_fp32_kernel(const float* __restrict__ in,
                                                                  const float* __restrict__ w,
                                                                  const float* __restrict__ bias,
                                                                  const float* resid,   // may alias out
                                                                  const int32_t* __restrict__ count,
                                                                  float* out) {
    extern __shared__ float sm[];   // [121][128]
    int row = blockIdx.x;
    if (row >= *count) return;
    for (int i = threadIdx.x; i < 121 * 32; i += F32_THREADS) reinterpret_cast<float4*>(sm)[i] = make_float4(0, 0, 0, 0);
    __syncthreads();
    const float4* src = reinterpret_cast<const float4*>(in + (size_t)row * 81 * 128);
    for (int i = threadIdx.x; i < 81 * 32; i += F32_THREADS) {
        int cell = i >> 5, q = i & 31;
        int r = cell / 9, c = cell - 9 * r;
        reinterpret_cast<float4*>(sm)[((r + 1) * 11 + (c + 1)) * 32 + q] = src[i];
    }
    __syncthreads();

    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int MAXC = 11;                  // ceil(81/8)
    float4 acc[MAXC];
    int base[MAXC];
#pragma unroll
    for (int j = 0; j < MAXC; j++) {
        acc[j] = make_float4(0, 0, 0, 0);
        int cell = warp + 8 * j;
        int cc = cell < 81 ? cell : 80;
        base[j] = ((cc / 9) * 11 + (cc % 9)) * 128;      // top-left tap of this cell in the padded tile
    }
    const float4* w4 = reinterpret_cast<const float4*>(w);
    for (int tap = 0; tap < 9; tap++) {
        int toff = ((tap / 3) * 11 + (tap % 3)) * 128;
        const float4* wt = w4 + (size_t)tap * 128 * 32 + lane;
#pragma unroll 4
        for (int ci = 0; ci < 128; ci++) {
            float4 wv = __ldg(wt + ci * 32);
#pragma unroll
            for (int j = 0; j < MAXC; j++) {
                float x = sm[base[j] + toff + ci];
                acc[j].x = fmaf(x, wv.x, acc[j].x);
                acc[j].y = fmaf(x, wv.y, acc[j].y);
                acc[j].z = fmaf(x, wv.z, acc[j].z);
                acc[j].w = fmaf(x, wv.w, acc[j].w);
            }
        }
    }
    float4 bv = reinterpret_cast<const float4*>(bias)[lane];
#pragma unroll
    for (int j = 0; j < MAXC; j++) {
        int cell = warp + 8 * j;
        if (cell < 81) {
            size_t o = ((size_t)row * 81 + cell) * 32 + lane;
            float4 v = make_float4(acc[j].x + bv.x, acc[j].y + bv.y, acc[j].z + bv.z, acc[j].w + bv.w);
            if (resid) {
                float4 rr = reinterpret_cast<const float4*>(resid)[o];
                v.x += rr.x; v.y += rr.y; v.z += rr.z; v.w += rr.w;
            }
            v.x = fmaxf(v.x, 0.0f); v.y = fmaxf(v.y, 0.0f); v.z = fmaxf(v.z, 0.0f); v.w = fmaxf(v.w, 0.0f);
            reinterpret_cast<float4*>(out)[o] = v;
        }
    }
}

// ---------------------------------------------------------------- heads (dual_network.py:101-119)
// One block (128 threads) per position. act: [row][81][128] fp32 or bf16.
__global__ void __launch_bounds__(128) heads_kernel(NetWeights W, const float* __restrict__ act_f32,
                                                    const __nv_bfloat16* __restrict__ act_bf16,
                                                    const int32_t* __restrict__ count, float* __restrict__ policy,
                                                    float* __restrict__ value, int row_stride) {
    int row = blockIdx.x;
    if (row >= *count) return;
    __shared__ float ph[162];     // policy head feature map, CHW flatten: j*81 + cell
    __shared__ float vh[81];
    __shared__ float hid[256];
    __shared__ float red[4];
    __shared__ float logit[81];
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // head_w: policy conv [2][128], value conv [128], their BN shifts [384..386]
    float wp0[4], wp1[4], wv[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        wp0[i] = W.head_w[lane * 4 + i];
        wp1[i] = W.head_w[128 + lane * 4 + i];
        wv[i] = W.head_w[256 + lane * 4 + i];
    }
    for (int cell = warp; cell < 81; cell += 4) {
        float x[4];
        size_t o = ((size_t)row * 81 + cell) * 128 + lane * 4;
        if (act_f32) {
            float4 v = *reinterpret_cast<const float4*>(act_f32 + o);
            x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
        } else {
            uint2 v = *reinterpret_cast<const uint2*>(act_bf16 + o);
            __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&v.x), b = *reinterpret_cast<__nv_bfloat162*>(&v.y);
            x[0] = __low2float(a); x[1] = __high2float(a); x[2] = __low2float(b); x[3] = __high2float(b);
        }
        float s0 = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < 4; i++) { s0 = fmaf(x[i], wp0[i], s0); s1 = fmaf(x[i], wp1[i], s1); s2 = fmaf(x[i], wv[i], s2); }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            s0 += __shfl_xor_sync(0xFFFFFFFFu, s0, off);
            s1 += __shfl_xor_sync(0xFFFFFFFFu, s1, off);
            s2 += __shfl_xor_sync(0xFFFFFFFFu, s2, off);
        }
        if (lane == 0) {
            ph[cell] = fmaxf(s0 + W.head_w[384], 0.0f);
            ph[81 + cell] = fmaxf(s1 + W.head_w[385], 0.0f);
            vh[cell] = fmaxf(s2 + W.head_w[386], 0.0f);
        }
    }
    __syncthreads();
    // policy FC (162 -> 81), weights transposed [162][81]
    float lg = -INFINITY;
    if (threadIdx.x < 81) {
        float a = W.pol_fc_b[threadIdx.x];
        for (int i = 0; i < 162; i++) a = fmaf(ph[i], W.pol_fc_w[i * 81 + threadIdx.x], a);
        lg = a;
        logit[threadIdx.x] = a;
    }
    // value FC1 (81 -> 256), weights transposed [81][256]
    for (int j = threadIdx.x; j < 256; j += 128) {
        float a = W.val_fc1_b[j];
        for (int i = 0; i < 81; i++) a = fmaf(vh[i], W.val_fc1_w[i * 256 + j], a);
        hid[j] = fmaxf(a, 0.0f);
    }
    // softmax over the 81 logits (dual_network.py:108)
    float m = lg;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, off));
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
    float e = (threadIdx.x < 81) ? expf(lg - m) : 0.0f;
    float s = e;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, off);
    __syncthreads();
    if (lane == 0) red[warp] = s;
    __syncthreads();
    s = red[0] + red[1] + red[2] + red[3];
    size_t orow = (size_t)row * row_stride;
    if (threadIdx.x < 81) policy[orow * 81 + threadIdx.x] = e / s;
    // value FC2 (256 -> 1) + tanh (dual_network.py:118-119)
    float a = hid[threadIdx.x] * W.val_fc2_w[threadIdx.x] + hid[threadIdx.x + 128] * W.val_fc2_w[threadIdx.x + 128];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xFFFFFFFFu, a, off);
    __syncthreads();
    if (lane == 0) red[warp] = a;
    __syncthreads();
    if (threadIdx.x == 0) value[orow] = tanhf(red[0] + red[1] + red[2] + red[3] + W.val_fc2_b[0]);
}

// Heads after the tensor-core trunk when they are not fused into its tail (batches of more than one group per CTA
// pair, the single-CTA trunks, uttt_net_forward on large batches): one block per HEADS_P positions, see heads_fc.cuh.
__global__ void __launch_bounds__(HEADS_THREADS) heads_fc_kernel(HeadsFC W, const float* __restrict__ headfeat,
                                                                 const int32_t* __restrict__ count, float* __restrict__ policy,
                                                                 float* __restrict__ value, int row_stride) {
    pdl_trigger();          // (programmatic dependent launch, common.cuh: the next kernel of the round loop may be scheduled)
    pdl_wait();             // the trunk kernel has finished: its head features are visible
    const int row0 = blockIdx.x * HEADS_P;
    const int n = *count;
    if (row0 >= n) return;
    extern __shared__ __align__(16) float heads_sm[];
    heads_fc_block(W, headfeat, row0, 1, min(HEADS_P, n - row0), policy, value, row_stride, heads_sm);
}

cudaError_t net_fp32_init() {
    cudaError_t e = cudaFuncSetAttribute(heads_fc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HEADS_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(conv3x3_fp32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, F32_SMEM);
}

cudaError_t launch_heads_fc(const NetWeights& w, const float* headfeat, const int32_t* count, int max_rows, float* policy,
                            float* value, int row_stride, cudaStream_t s) {
    return launch_pdl(heads_fc_kernel, dim3((max_rows + HEADS_P - 1) / HEADS_P), dim3(HEADS_THREADS), HEADS_SMEM_BYTES, s, heads_fc_of(w),
                      headfeat, count, policy, value, row_stride);
}

cudaError_t launch_conv_input(const NetWeights& w, const __nv_bfloat16* planes, const int32_t* count, int max_rows,
                              float* out, cudaStream_t s) {
    conv_input_kernel<<<max_rows, 128, 0, s>>>(planes, w.conv_in_w, w.conv_in_b, count, out);
    return cudaGetLastError();
}

cudaError_t launch_trunk_fp32(const NetWeights& w, const __nv_bfloat16* planes, const int32_t* count, int max_rows,
                              float* act_a, float* act_b, cudaStream_t s) {
    cudaError_t e = launch_conv_input(w, planes, count, max_rows, act_a, s);
    if (e != cudaSuccess) return e;
    // residual block: a --conv1--> b --conv2(+a)--> a          dual_network.py:36-45
    for (int blk = 0; blk < NET_BLOCKS; blk++) {
        const float* w1 = w.res_w + (size_t)(2 * blk) * 9 * 128 * 128;
        const float* w2 = w.res_w + (size_t)(2 * blk + 1) * 9 * 128 * 128;
        conv3x3_fp32_kernel<<<max_rows, F32_THREADS, F32_SMEM, s>>>(act_a, w1, w.res_b + (2 * blk) * 128, nullptr, count, act_b);
        conv3x3_fp32_kernel<<<max_rows, F32_THREADS, F32_SMEM, s>>>(act_b, w2, w.res_b + (2 * blk + 1) * 128, act_a, count, act_a);
    }
    return cudaGetLastError();
}

cudaError_t launch_heads(const NetWeights& w, const float* act_f32, const __nv_bfloat16* act_bf16, const int32_t* count,
                         int max_rows, float* policy, float* value, int row_stride, cudaStream_t s) {
    heads_kernel<<<max_rows, 128, 0, s>>>(w, act_f32, act_bf16, count, policy, value, row_stride);
    return cudaGetLastError();
}

}  // namespace uttt
