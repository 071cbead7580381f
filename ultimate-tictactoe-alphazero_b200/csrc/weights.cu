// weights.cu -- the network weights on the device: eval-mode BatchNorm folding and every layout the kernels read, in
// one allocation per engine (NetWeights, common.cuh).
//
// The residual convolutions (4.7 M weights) are folded and packed on the device by pack_res_kernel; conv_input, the
// BatchNorm shifts as tensor-core bias blocks, and the heads are built on the host into an image of the first part of
// the block and uploaded with one copy.
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <type_traits>
#include <vector>

#include "common.cuh"
#include "heads_fc.cuh"
#include "tc_common.cuh"

namespace uttt {
namespace {

constexpr size_t N_RES = (size_t)NET_LAYERS * 9 * NET_C * NET_C, N_RES_BN = (size_t)NET_LAYERS * 4 * NET_C;
constexpr size_t BLK = 2 * 128 * 8;        // bf16 elements of one K = 16 tensor-core B block: [2 k-panels][128 co][8]

// The per-CTA halves of a B operand for cta_group::2 MMAs: each CTA of a pair holds the output channels
// 64*rank .. 64*rank+63, and its share of a weight stage of `bps` blocks is one contiguous bulk copy.
// [block b][sub][2 k-panels][128 co][8] -> [stage][cta rank][block of the stage][sub][2 k-panels][64 co][8], with `subs`
// parts per block (2 for the split-bf16 arrays: hi, lo).  Returns the index of the 16-byte unit (co, 8 k).
__host__ __device__ __forceinline__ size_t half_unit(int b, int sub, int pnl, int co, int bps, int subs) {
    const int stage = b / bps, j = b - stage * bps;
    return (((((size_t)stage * 2 + (co >> 6)) * bps + j) * subs + sub) * 2 + pnl) * 64 + (co & 63);
}

// Folding and packing of the 32 residual 3x3 convolutions: raw (32)(co,ci,ky,kx) fp32 + bn (32)(4)(128) ->
// fp32 [l][tap][ci][co] and shift [l][co], and bf16 blocks [l][K-block][ci/8 % 2][co][ci%8] (K-blocks in the order of
// tcx::kblock_of) as per-CTA halves in stages of 8 and 18 blocks and, with lo = bf16(w - hi), of 6 blocks.
__global__ void __launch_bounds__(256) pack_res_kernel(NetWeights w) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;      // index into raw
    if (i >= N_RES) return;
    int tap = (int)(i % 9);
    size_t r = i / 9;
    int ci = (int)(r % 128);
    r /= 128;
    int co = (int)(r % 128);
    int l = (int)(r / 128);
    const float* b = w.raw_res_bn + (size_t)l * 4 * 128;
    float g = b[co], beta = b[128 + co], m = b[256 + co], v = b[384 + co];
    float sc = __fdiv_rn(g, __fsqrt_rn(__fadd_rn(v, 1e-5f)));
    float val = __fmul_rn(w.raw_res[i], sc);
    w.res_w[(((size_t)l * 9 + tap) * 128 + ci) * 128 + co] = val;
    const int blk = l * 72 + tcx::kblock_of(tap, ci / 16), pnl = (ci / 8) & 1, k = ci % 8;
    const __nv_bfloat16 hi = __float2bfloat16(val);
    w.res_w_2sm[half_unit(blk, 0, pnl, co, 8, 1) * 8 + k] = hi;
    w.res_w_2sm18[half_unit(blk, 0, pnl, co, 18, 1) * 8 + k] = hi;
    w.res_w_x3p[half_unit(blk, 0, pnl, co, 6, 2) * 8 + k] = hi;
    w.res_w_x3p[half_unit(blk, 1, pnl, co, 6, 2) * 8 + k] = __float2bfloat16(__fsub_rn(val, __bfloat162float(hi)));
    if (ci == 0 && tap == 0) w.res_b[l * 128 + co] = __fsub_rn(beta, __fmul_rn(m, sc));
}

// The table of the block: every array with its number of elements, each at a multiple of 256 bytes (where a cudaMalloc
// of its own would place it).  The arrays built on the host come first, `host_bytes` of them; then the staging of the
// caller's residual tensors and what pack_res_kernel writes.  Points w's arrays into the block at `base`; returns its size.
size_t carve(NetWeights& w, uintptr_t base, size_t& host_bytes) {
    size_t off = 0;
    auto at = [&](auto*& p, size_t n) {
        p = reinterpret_cast<std::remove_reference_t<decltype(p)>>(base + off);
        off += (n * sizeof(*p) + 255) / 256 * 256;
    };
    at(w.conv_in_w, 9 * 3 * 128); at(w.conv_in_b, 128);
    at(w.conv_in_w_2sm, 16 * BLK); at(w.conv_in_w_2sm18, 18 * BLK); at(w.conv_in_w_x3p, 12 * 2 * BLK);
    at(w.bias_blk_2sm, 33 * BLK); at(w.bias_blk_x3p, 33 * BLK);
    at(w.head_w, 387); at(w.heads_pack, HEADS_PACK_FLOATS);
    at(w.pol_fc_w, 162 * 81); at(w.pol_fc_b, 81); at(w.val_fc1_w, 81 * 256); at(w.val_fc1_b, 256);
    at(w.val_fc2_w, 256); at(w.val_fc2_b, 1);
    host_bytes = off;
    at(w.raw_res, N_RES); at(w.raw_res_bn, N_RES_BN);
    at(w.res_w, N_RES); at(w.res_b, NET_LAYERS * 128);
    at(w.res_w_2sm, N_RES); at(w.res_w_2sm18, N_RES); at(w.res_w_x3p, 2 * N_RES);
    return off;
}

// Eval-mode BatchNorm folding: y = gamma*(x-mean)/sqrt(var+eps) + beta = scale*x + shift.
void bn_fold(const float* bn, int C, std::vector<float>& scale, std::vector<float>& shift) {
    scale.resize(C); shift.resize(C);
    for (int c = 0; c < C; c++) {
        float g = bn[c], b = bn[C + c], m = bn[2 * C + c], v = bn[3 * C + c];
        float s = g / sqrtf(v + 1e-5f);
        scale[c] = s;
        shift[c] = b - m * s;
    }
}

}  // namespace

int upload_weights(NetWeights& W, const uttt_weights* w, int on_device, const float* const* res_tab,
                   const float* const (*res_bn_tab)[4], cudaStream_t s) {
    size_t host_bytes;
    if (!W.block) {
        const size_t bytes = carve(W, 0, host_bytes);
        UTTT_CUDA_OK(cudaMalloc((void**)&W.block, bytes));
        UTTT_CUDA_OK(cudaMemset(W.block, 0, bytes));
    }
    carve(W, (uintptr_t)W.block, host_bytes);

    // what is not built by pack_res_kernel is built on the host in `img`, the image of the block's first host_bytes
    std::vector<uint8_t> img(host_bytes);
    auto host = [&](auto* dev) { return reinterpret_cast<decltype(dev)>(img.data() + ((uint8_t*)dev - W.block)); };
    auto fetch = [&](const float* p, size_t n, float* dst) -> int {
        UTTT_CHECK(p != nullptr, "null weight tensor");
        if (on_device) UTTT_CUDA_OK(cudaMemcpy(dst, p, n * sizeof(float), cudaMemcpyDeviceToHost));
        else memcpy(dst, p, n * sizeof(float));
        return 0;
    };
    std::vector<float> ciw(128 * 27), bni(4 * 128), pcw(2 * 128), pbn(8), pfw(81 * 162), vcw(128), vbn(4), v1w(256 * 81);
    if (fetch(w->conv_input_w, ciw.size(), ciw.data()) || fetch(w->bn_input, bni.size(), bni.data()) ||
        fetch(w->policy_conv_w, pcw.size(), pcw.data()) || fetch(w->policy_bn, pbn.size(), pbn.data()) ||
        fetch(w->policy_fc_w, pfw.size(), pfw.data()) || fetch(w->policy_fc_b, 81, host(W.pol_fc_b)) ||
        fetch(w->value_conv_w, vcw.size(), vcw.data()) || fetch(w->value_bn, vbn.size(), vbn.data()) ||
        fetch(w->value_fc1_w, v1w.size(), v1w.data()) || fetch(w->value_fc1_b, 256, host(W.val_fc1_b)) ||
        fetch(w->value_fc2_w, 256, host(W.val_fc2_w)) || fetch(w->value_fc2_b, 1, host(W.val_fc2_b)))
        return 1;

    // the 32 residual convolutions: staged in the block as they are, folded and packed by a kernel
    if (res_tab) {
        const size_t per = (size_t)128 * 128 * 9;
        for (int l = 0; l < 32; l++) {
            UTTT_CHECK(res_tab[l] != nullptr, "null weight tensor");
            // (cudaMemcpyDefault: each tensor may lie in host or device memory, whatever `on_device` says about `small`)
            UTTT_CUDA_OK(cudaMemcpyAsync(W.raw_res + l * per, res_tab[l], per * sizeof(float), cudaMemcpyDefault, s));
            for (int j = 0; j < 4; j++) {
                UTTT_CHECK(res_bn_tab[l][j] != nullptr, "null weight tensor");
                UTTT_CUDA_OK(cudaMemcpyAsync(W.raw_res_bn + (l * 4 + j) * 128, res_bn_tab[l][j], 128 * sizeof(float),
                                             cudaMemcpyDefault, s));
            }
        }
    } else {
        UTTT_CHECK(w->res_conv_w && w->res_bn, "null weight tensor");
        const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        UTTT_CUDA_OK(cudaMemcpyAsync(W.raw_res, w->res_conv_w, N_RES * sizeof(float), kind, s));
        UTTT_CUDA_OK(cudaMemcpyAsync(W.raw_res_bn, w->res_bn, N_RES_BN * sizeof(float), kind, s));
    }
    pack_res_kernel<<<ceil_div((int64_t)N_RES, 256), 256, 0, s>>>(W);
    UTTT_CUDA_OK(cudaGetLastError());

    // conv_input: (128,3,3,3) [co][ci][ky][kx] -> fp32 [tap][ci][co]; for the tensor pipe a layer of K = 16 per tap in
    // the bf16 layouts and split bf16 (input channels 3..15 and the tap slots past the 9th stay zero)
    std::vector<float> sc, sh;
    bn_fold(bni.data(), 128, sc, sh);
    float* ci_w = host(W.conv_in_w);
    memcpy(host(W.conv_in_b), sh.data(), 128 * sizeof(float));
    __nv_bfloat16 *c8 = host(W.conv_in_w_2sm), *c18 = host(W.conv_in_w_2sm18), *cx3 = host(W.conv_in_w_x3p);
    for (int co = 0; co < 128; co++)
        for (int ci = 0; ci < 3; ci++)
            for (int tap = 0; tap < 9; tap++) {
                const float v = ciw[(co * 3 + ci) * 9 + tap] * sc[co];
                ci_w[(tap * 3 + ci) * 128 + co] = v;
                const __nv_bfloat16 hi = __float2bfloat16(v);
                c8[half_unit(tap, 0, 0, co, 8, 1) * 8 + ci] = hi;
                c18[half_unit(tap, 0, 0, co, 18, 1) * 8 + ci] = hi;
                cx3[half_unit(tap, 0, 0, co, 6, 2) * 8 + ci] = hi;
                cx3[half_unit(tap, 1, 0, co, 6, 2) * 8 + ci] = __float2bfloat16(v - __bfloat162float(hi));
            }

    // heads: 1x1 convolutions with the BN scale folded in, and the FC weights transposed to [in][out]
    float* hw = host(W.head_w);
    bn_fold(pbn.data(), 2, sc, sh);
    for (int j = 0; j < 2; j++)
        for (int c = 0; c < 128; c++) hw[j * 128 + c] = pcw[j * 128 + c] * sc[j];
    hw[384] = sh[0]; hw[385] = sh[1];
    bn_fold(vbn.data(), 1, sc, sh);
    for (int c = 0; c < 128; c++) hw[256 + c] = vcw[c] * sc[0];
    hw[386] = sh[0];
    float *pf_t = host(W.pol_fc_w), *v1_t = host(W.val_fc1_w);
    for (int o = 0; o < 81; o++)
        for (int i = 0; i < 162; i++) pf_t[i * 81 + o] = pfw[o * 162 + i];
    for (int j = 0; j < 256; j++)
        for (int i = 0; i < 81; i++) v1_t[i * 256 + j] = v1w[j * 81 + i];
    // FC weights of the heads in the order heads_fc_block streams them: 3 chunks of 27 input rows
    for (int c = 0; c < HEADS_CHUNKS; c++) {
        float* dst = host(W.heads_pack) + (size_t)c * HEADS_CHUNK_FLOATS;
        for (int h = 0; h < 2; h++)
            for (int i = 0; i < HEADS_CHUNK_ROWS; i++)
                for (int o = 0; o < 81; o++)
                    dst[h * HEADS_POL_FLOATS + i * 81 + o] = pf_t[(size_t)(h * 81 + c * HEADS_CHUNK_ROWS + i) * 81 + o];
        for (int i = 0; i < HEADS_CHUNK_ROWS; i++)
            for (int j = 0; j < 256; j++)
                dst[2 * HEADS_POL_FLOATS + i * 256 + j] = v1_t[(size_t)(c * HEADS_CHUNK_ROWS + i) * 256 + j];
    }

    // bias blocks of the tensor-core trunks for conv_input's shift and the 32 residual layers' (from pack_res_kernel):
    // the shift as a sum of bf16 terms, multiplied by a constant A row -- hi, lo (k = 0, 1) for the bf16 trunks, three
    // terms (k = 0, 1, 2) for the split-bf16 one
    std::vector<float> shift(33 * 128);
    memcpy(shift.data(), host(W.conv_in_b), 128 * sizeof(float));
    UTTT_CUDA_OK(cudaMemcpyAsync(shift.data() + 128, W.res_b, 32 * 128 * sizeof(float), cudaMemcpyDeviceToHost, s));
    UTTT_CUDA_OK(cudaStreamSynchronize(s));
    __nv_bfloat16 *bb2 = host(W.bias_blk_2sm), *bx3 = host(W.bias_blk_x3p);
    for (int l = 0; l < 33; l++)
        for (int co = 0; co < 128; co++) {
            float b = shift[l * 128 + co];
            for (int k = 0; k < 3; k++) {
                const __nv_bfloat16 t = __float2bfloat16(b);
                if (k < 2) bb2[half_unit(l, 0, 0, co, 1, 1) * 8 + k] = t;
                bx3[half_unit(l, 0, 0, co, 1, 1) * 8 + k] = t;
                b -= __bfloat162float(t);
            }
        }
    UTTT_CUDA_OK(cudaMemcpyAsync(W.block, img.data(), host_bytes, cudaMemcpyHostToDevice, s));
    UTTT_CUDA_OK(cudaStreamSynchronize(s));
    W.loaded = true;
    return 0;
}

void release_weights(NetWeights& w) {
    cudaFree(w.block);
    w = NetWeights{};
}

}  // namespace uttt
