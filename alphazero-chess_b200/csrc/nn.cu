// Policy/value network of agent.rs:11-144 on the device.
//   bf16 path : 21 tcgen05 3x3 convolutions (nn_tc.cu) + one fused head kernel
//   fp32 path : straightforward fp32 kernels (parity mode, 1e-5 against a torch fp32 reference)
// BatchNorm (inference form, eps = 1e-5) is folded into the preceding convolution when the weights are imported.
#include "nn.h"
#include "nn_tc.h"
#include "device_once.h"
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <vector>

namespace azb {

// ---------------------------------------------------------------------------------------------- weight catalogue
static const int kBlocks = 10;
static int64_t weight_size(int i) {
    if (i == 0) return 128 * 19 * 9;
    if (i < 6) return 128;
    i -= 6;
    if (i < kBlocks * 12) { int j = i % 12; return (j == 0 || j == 6) ? 128 * 128 * 9 : 128; }
    i -= kBlocks * 12;
    static const int64_t tail[18] = {32 * 128, 32, 32, 32, 32, 32, 64 * 32, 64, 8 * 128, 8, 8, 8, 8, 8, 512 * 64, 64, 64, 1};
    return i < 18 ? tail[i] : 0;
}
static std::string weight_name(int i) {
    static const char* bn[4] = {"gamma", "beta", "running_mean", "running_var"};
    if (i == 0) return "input_conv.weight";
    if (i == 1) return "input_conv.bias";
    if (i < 6) return std::string("input_bn.") + bn[i - 2];
    i -= 6;
    if (i < kBlocks * 12) {
        int b = i / 12, j = i % 12;
        std::string p = "res_blocks." + std::to_string(b) + ".";
        int half = j / 6, k = j % 6;
        std::string c = half ? "conv2" : "conv1", n = half ? "bn2" : "bn1";
        if (k == 0) return p + c + ".weight";
        if (k == 1) return p + c + ".bias";
        return p + n + "." + bn[k - 2];
    }
    i -= kBlocks * 12;
    static const char* tail[18] = {"policy_conv_1.weight", "policy_conv_1.bias", "policy_bn.gamma", "policy_bn.beta",
                                   "policy_bn.running_mean", "policy_bn.running_var", "policy_conv_2.weight", "policy_conv_2.bias",
                                   "value_conv.weight", "value_conv.bias", "value_bn.gamma", "value_bn.beta", "value_bn.running_mean",
                                   "value_bn.running_var", "value_linear_1.weight", "value_linear_1.bias", "value_linear_2.weight",
                                   "value_linear_2.bias"};
    return i < 18 ? tail[i] : "";
}

template <class T>
static int dmalloc(az_engine* e, T** p, size_t n) {
    return check_cuda(e, cudaMalloc(p, n * sizeof(T)), "cudaMalloc(net)");
}

// the weights of one network (fp32 parameters, bf16 operands) and their tensor maps
static int alloc_weights(az_engine* e, NetWeights* w) {
    int r = 0;
    r |= dmalloc(e, &w->f_w_in, 128 * 19 * 9); r |= dmalloc(e, &w->f_b_in, 128);
    r |= dmalloc(e, &w->f_w_tower, (size_t)20 * 128 * 128 * 9); r |= dmalloc(e, &w->f_b_tower, 21 * 128);  // row 20: copy of f_b_in for the fused launch
    r |= dmalloc(e, &w->f_w40t, 128 * 40); r |= dmalloc(e, &w->f_b40, 40);
    r |= dmalloc(e, &w->f_wp2t, 32 * 64); r |= dmalloc(e, &w->f_bp2, 64);
    r |= dmalloc(e, &w->f_wl1, 512 * 64); r |= dmalloc(e, &w->f_bl1, 64);
    r |= dmalloc(e, &w->f_wl2, 64); r |= dmalloc(e, &w->f_bl2, 1);
    const int ic = w->in_ch;
    r |= dmalloc(e, &w->h_w_in, (size_t)9 * 128 * ic); r |= dmalloc(e, &w->h_w_tower, (size_t)20 * 9 * 128 * 128);
    r |= dmalloc(e, &w->h_w40, 40 * 128); r |= dmalloc(e, &w->h_wp2, 64 * 32); r |= dmalloc(e, &w->h_wl1t, 64 * 512);
    if (r) return AZ_ERR_OUT_OF_MEMORY;
    if (tc_make_weight_map(&w->map_w_in, w->h_w_in, ic)) return set_err(e, AZ_ERR_CUDA, "cuTensorMapEncodeTiled(w_in)");
    for (int l = 0; l < 20; l++)
        if (tc_make_weight_map(&w->map_w_tower[l], w->h_w_tower + (size_t)l * 9 * 128 * 128, 128))
            return set_err(e, AZ_ERR_CUDA, "cuTensorMapEncodeTiled(w_tower)");
    return 0;
}

int net_create(az_engine* e) {
    NetWeights* w = new NetWeights;
    e->net = w;
    w->max_boards = e->max_batch;
    const size_t nb = (size_t)e->max_batch;
    w->in_ch = e->knobs.input_k32 ? 32 : 64;
    const int ic = w->in_ch;
    int r = alloc_weights(e, w);
    if (r) return r;
    r |= dmalloc(e, &w->a_in, nb * 64 * ic);
    for (int i = 0; i < 3; i++) r |= dmalloc(e, &w->a_buf[i], nb * 64 * 128);
    if (r) return AZ_ERR_OUT_OF_MEMORY;
    cudaMemset(w->a_in, 0, nb * 64 * ic * 2);
    if (tc_make_act_map(&w->map_a_in, w->a_in, ic, e->max_batch)) return set_err(e, AZ_ERR_CUDA, "cuTensorMapEncodeTiled(a_in)");
    for (int i = 0; i < 3; i++)
        if (tc_make_act_map(&w->map_a[i], w->a_buf[i], 128, e->max_batch)) return set_err(e, AZ_ERR_CUDA, "cuTensorMapEncodeTiled(act)");
    for (int i = 0; i < 3; i++)
        if (tc_make_rows_map(&w->map_rows[i], w->a_buf[i], e->max_batch)) return set_err(e, AZ_ERR_CUDA, "cuTensorMapEncodeTiled(rows)");
    CUtensorMap host_maps[31];
    for (int i = 0; i < 3; i++) host_maps[i] = w->map_a[i];
    for (int l = 0; l < 20; l++) host_maps[3 + l] = w->map_w_tower[l];
    host_maps[23] = w->map_a_in;
    host_maps[24] = w->map_w_in;
    for (int i = 0; i < 3; i++)   // 16-file boxes for the wide tower (AZ_TOWER_WIDE)
        if (tc_make_act_map(&host_maps[25 + i], w->a_buf[i], 128, e->max_batch, 1)) return set_err(e, AZ_ERR_CUDA, "cuTensorMapEncodeTiled(act, wide)");
    for (int i = 0; i < 3; i++)   // 10-file boxes (AZ_TOWER_WIDE=2)
        if (tc_make_act_map(&host_maps[28 + i], w->a_buf[i], 128, e->max_batch, 2)) return set_err(e, AZ_ERR_CUDA, "cuTensorMapEncodeTiled(act, wide 2)");
    if (dmalloc(e, &w->d_maps, 31)) return AZ_ERR_OUT_OF_MEMORY;
    AZ_CUDA(e, cudaMemcpy(w->d_maps, host_maps, sizeof host_maps, cudaMemcpyHostToDevice));
    return 0;
}

// Network slot 1: its own weights, tensor maps and device map array (the activation maps of slot 0, its weight maps); the
// activations and every other buffer stay slot 0's
static int create_slot1(az_engine* e) {
    NetWeights* w0 = e->net;
    NetWeights* w = new NetWeights;
    e->net1 = w;
    w->max_boards = w0->max_boards;
    w->in_ch = w0->in_ch;
    int r = alloc_weights(e, w);
    if (r) return r;
    CUtensorMap host_maps[31];
    AZ_CUDA(e, cudaMemcpy(host_maps, w0->d_maps, sizeof host_maps, cudaMemcpyDeviceToHost));
    for (int l = 0; l < 20; l++) host_maps[3 + l] = w->map_w_tower[l];
    host_maps[24] = w->map_w_in;
    if (dmalloc(e, &w->d_maps, 31)) return AZ_ERR_OUT_OF_MEMORY;
    AZ_CUDA(e, cudaMemcpy(w->d_maps, host_maps, sizeof host_maps, cudaMemcpyHostToDevice));
    return 0;
}

NetWeights* net_slot(az_engine* e, int s) { return s == 0 ? e->net : s == 1 ? e->net1 : nullptr; }

void net_destroy(az_engine* e) {
    for (NetWeights** slot : {&e->net, &e->net1}) {
        NetWeights* w = *slot;
        if (!w) continue;
        cudaFree(w->f_w_in); cudaFree(w->f_b_in); cudaFree(w->f_w_tower); cudaFree(w->f_b_tower); cudaFree(w->f_w40t); cudaFree(w->f_b40);
        cudaFree(w->f_wp2t); cudaFree(w->f_bp2); cudaFree(w->f_wl1); cudaFree(w->f_bl1); cudaFree(w->f_wl2); cudaFree(w->f_bl2);
        cudaFree(w->d_maps);
        cudaFree(w->h_w_in); cudaFree(w->h_w_tower); cudaFree(w->a_in); cudaFree(w->h_w40); cudaFree(w->h_wp2); cudaFree(w->h_wl1t);
        for (int i = 0; i < 3; i++) { cudaFree(w->a_buf[i]); cudaFree(w->g_buf[i]); }
        delete w;
        *slot = nullptr;
    }
    cudaFree(e->d_net_counts); cudaFree(e->d_net_slot); cudaFree(e->d_net_value);
    e->d_net_counts = nullptr; e->d_net_slot = nullptr; e->d_net_value = nullptr;
}

// fold BN(gamma, beta, mean, var) into conv (weight [co][k], bias [co])
static void fold(const float* wt, const float* bias, const float* g, const float* b, const float* m, const float* v, int co, int k,
                 float* w_out, float* b_out) {
    for (int o = 0; o < co; o++) {
        float s = g[o] / std::sqrt(v[o] + 1e-5f);
        for (int i = 0; i < k; i++) w_out[(size_t)o * k + i] = wt[(size_t)o * k + i] * s;
        b_out[o] = (bias[o] - m[o]) * s + b[o];
    }
}

static int upload(az_engine* e, void* dst, const void* src, size_t bytes) {
    return check_cuda(e, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, e->stream), "upload weights");
}

static int load_from_host(az_engine* e, NetWeights* w, const float* const* a) {
    std::vector<float> fw((size_t)128 * 128 * 9), fb(128);
    std::vector<__nv_bfloat16> hw((size_t)9 * 128 * 128);
    int r = 0;
    // input conv: [128][19][3][3]
    fold(a[0], a[1], a[2], a[3], a[4], a[5], 128, 19 * 9, fw.data(), fb.data());
    r |= upload(e, w->f_w_in, fw.data(), 128 * 19 * 9 * 4);
    r |= upload(e, w->f_b_in, fb.data(), 128 * 4);
    r |= upload(e, w->f_b_tower + 20 * 128, fb.data(), 128 * 4);
    const int ic = w->in_ch;
    for (int tap = 0; tap < 9; tap++)
        for (int co = 0; co < 128; co++)
            for (int ci = 0; ci < ic; ci++)
                hw[((size_t)tap * 128 + co) * ic + ci] = __float2bfloat16_rn(ci < 19 ? fw[((size_t)co * 19 + ci) * 9 + tap] : 0.0f);
    r |= upload(e, w->h_w_in, hw.data(), (size_t)9 * 128 * ic * 2);
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    for (int l = 0; l < 20; l++) {
        const int o = 6 + (l / 2) * 12 + (l % 2) * 6;
        fold(a[o], a[o + 1], a[o + 2], a[o + 3], a[o + 4], a[o + 5], 128, 128 * 9, fw.data(), fb.data());
        r |= upload(e, w->f_w_tower + (size_t)l * 128 * 128 * 9, fw.data(), (size_t)128 * 128 * 9 * 4);
        r |= upload(e, w->f_b_tower + l * 128, fb.data(), 128 * 4);
        for (int tap = 0; tap < 9; tap++)
            for (int co = 0; co < 128; co++)
                for (int ci = 0; ci < 128; ci++)
                    hw[((size_t)tap * 128 + co) * 128 + ci] = __float2bfloat16_rn(fw[((size_t)co * 128 + ci) * 9 + tap]);
        r |= upload(e, w->h_w_tower + (size_t)l * 9 * 128 * 128, hw.data(), (size_t)9 * 128 * 128 * 2);
        AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    }
    const int h = 6 + kBlocks * 12;
    std::vector<float> w40(40 * 128), b40(40), w40t(128 * 40), wp2t(32 * 64);
    fold(a[h], a[h + 1], a[h + 2], a[h + 3], a[h + 4], a[h + 5], 32, 128, w40.data(), b40.data());
    fold(a[h + 8], a[h + 9], a[h + 10], a[h + 11], a[h + 12], a[h + 13], 8, 128, w40.data() + 32 * 128, b40.data() + 32);
    for (int o = 0; o < 40; o++) for (int c = 0; c < 128; c++) w40t[c * 40 + o] = w40[o * 128 + c];
    for (int o = 0; o < 64; o++) for (int c = 0; c < 32; c++) wp2t[c * 64 + o] = a[h + 6][o * 32 + c];
    r |= upload(e, w->f_w40t, w40t.data(), 128 * 40 * 4); r |= upload(e, w->f_b40, b40.data(), 40 * 4);
    r |= upload(e, w->f_wp2t, wp2t.data(), 32 * 64 * 4); r |= upload(e, w->f_bp2, a[h + 7], 64 * 4);
    r |= upload(e, w->f_wl1, a[h + 14], 512 * 64 * 4); r |= upload(e, w->f_bl1, a[h + 15], 64 * 4);
    r |= upload(e, w->f_wl2, a[h + 16], 64 * 4); r |= upload(e, w->f_bl2, a[h + 17], 4);
    std::vector<__nv_bfloat16> hw40(40 * 128), hwp2(64 * 32), hwl1t(64 * 512);
    for (int i = 0; i < 40 * 128; i++) hw40[i] = __float2bfloat16_rn(w40[i]);
    for (int i = 0; i < 64 * 32; i++) hwp2[i] = __float2bfloat16_rn(a[h + 6][i]);
    for (int o = 0; o < 64; o++) for (int i = 0; i < 512; i++) hwl1t[o * 512 + i] = __float2bfloat16_rn(a[h + 14][i * 64 + o]);
    r |= upload(e, w->h_w40, hw40.data(), 40 * 128 * 2); r |= upload(e, w->h_wp2, hwp2.data(), 64 * 32 * 2);
    r |= upload(e, w->h_wl1t, hwl1t.data(), 64 * 512 * 2);
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    if (r) return AZ_ERR_CUDA;
    w->loaded = true;
    return 0;
}

// ---------------------------------------------------------------------------------------------- plane converters
__global__ void k_planes_to_bf16(const float* __restrict__ planes, __nv_bfloat16* __restrict__ out, int n, int chunks) {
    // out [n][64 sq][ch]; one thread per (board, square, 8-channel chunk); chunks = ch / 8 (8 or 4)
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n * 64 * chunks) return;
    const int b = (int)(i / (size_t)(64 * chunks)), sq = (int)((i / chunks) & 63), chunk = (int)(i % chunks);
    uint32_t packed[4] = {0, 0, 0, 0};
    if (chunk < 3) {
        for (int j = 0; j < 8; j++) {
            int c = chunk * 8 + j;
            float v = c < AZ_NUM_PLANES ? planes[((size_t)b * AZ_NUM_PLANES + c) * 64 + sq] : 0.0f;
            __nv_bfloat16 h = __float2bfloat16_rn(v);
            packed[j >> 1] |= (uint32_t)(*reinterpret_cast<unsigned short*>(&h)) << ((j & 1) * 16);
        }
    }
    reinterpret_cast<uint4*>(out)[i] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
}
void launch_planes_to_bf16(cudaStream_t s, const float* planes, __nv_bfloat16* out, int n, int ch) {
    if (n > 0) k_planes_to_bf16<<<(unsigned)(((size_t)n * 8 * ch + 255) / 256), 256, 0, s>>>(planes, out, n, ch / 8);
}
__global__ void k_encode_bf16_wire(const az_position* __restrict__ wire, __nv_bfloat16* __restrict__ out, int n, int ch) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n) return;
    DPos p = dpos_from_wire(wire[warp]);
    encode_bf16_warp(p, out + (size_t)warp * 64 * ch, lane, ch);
}
void launch_encode_bf16_wire(cudaStream_t s, const az_position* wire, __nv_bfloat16* out, int n, int ch) {
    if (n > 0) k_encode_bf16_wire<<<(n + 3) / 4, 128, 0, s>>>(wire, out, n, ch);
}

// rows of a multi-network batch back in the caller's order: row i of the outputs is slot[i] of the batch (one block per row)
__global__ void k_gather_rows(const float* __restrict__ policy, const float* __restrict__ value, const int* __restrict__ slot,
                              float* __restrict__ policy_out, float* __restrict__ value_out) {
    const int i = blockIdx.x, s = slot[i];
    const float4* src = reinterpret_cast<const float4*>(policy + (size_t)s * AZ_ACTION_SPACE);
    float4* dst = reinterpret_cast<float4*>(policy_out + (size_t)i * AZ_ACTION_SPACE);
    for (int j = threadIdx.x; j < AZ_ACTION_SPACE / 4; j += blockDim.x) dst[j] = src[j];
    if (threadIdx.x == 0) value_out[i] = value[s];
}

// ---------------------------------------------------------------------------------------------- fp32 convolution
// NCHW fp32 3x3 same conv + bias (+residual) (+relu); one block per board, thread = (pixel, group of 32 out channels)
template <int CIN>
__global__ void __launch_bounds__(256) k_conv3x3_f32(const float* __restrict__ in, const float* __restrict__ wgt, const float* __restrict__ bias,
                                                     const float* __restrict__ residual, float* __restrict__ out, const int* __restrict__ n_dev,
                                                     int n_static, int relu) {
    extern __shared__ float xs[];  // [CIN][64]
    const int n = n_dev ? *n_dev : n_static;
    const int b = blockIdx.x;
    if (b >= n) return;
    for (int i = threadIdx.x; i < CIN * 64; i += 256) xs[i] = in[(size_t)b * CIN * 64 + i];
    __syncthreads();
    const int px = threadIdx.x & 63, cobase = (threadIdx.x >> 6) * 32;
    const int r = px >> 3, f = px & 7;
    float acc[32];
#pragma unroll
    for (int j = 0; j < 32; j++) acc[j] = bias[cobase + j];
    for (int ci = 0; ci < CIN; ci++) {
#pragma unroll
        for (int tap = 0; tap < 9; tap++) {
            const int rr = r + tap / 3 - 1, ff = f + tap % 3 - 1;
            const float x = (rr >= 0 && rr < 8 && ff >= 0 && ff < 8) ? xs[ci * 64 + rr * 8 + ff] : 0.0f;
            const float* wp = wgt + ((size_t)cobase * CIN + ci) * 9 + tap;
#pragma unroll
            for (int j = 0; j < 32; j++) acc[j] = fmaf(__ldg(wp + (size_t)j * CIN * 9), x, acc[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < 32; j++) {
        const size_t o = ((size_t)b * 128 + cobase + j) * 64 + px;
        float v = acc[j];
        if (residual) v += residual[o];
        if (relu) v = fmaxf(v, 0.0f);
        out[o] = v;
    }
}

// ---------------------------------------------------------------------------------------------- heads (fp32 path)
// One block (256 threads) per board: policy_conv_1+bn+relu and value_conv+bn+relu (40 x 128 per square),
// policy_conv_2 (64 x 32 per square), softmax over the 4096 logits, value MLP + tanh (agent.rs:124-141).
// Tower output NCHW f32 [b][128][64].  (The bf16 path uses the tensor-core kernel in nn_heads.cu.)
constexpr int HEAD_SMEM = (128 * 65 + 128 * 40 + 40 * 64 + 64) * 4;

__global__ void __launch_bounds__(256) k_heads_f32(const float* __restrict__ tower, const float* __restrict__ w40t, const float* __restrict__ b40,
                                               const float* __restrict__ wp2t, const float* __restrict__ bp2, const float* __restrict__ wl1,
                                               const float* __restrict__ bl1, const float* __restrict__ wl2, const float* __restrict__ bl2,
                                               float* __restrict__ policy_out, float* __restrict__ value_out, const int* __restrict__ n_dev,
                                               int n_static) {
    extern __shared__ float sm[];
    float* xs = sm;                  // [128][65] channel-major (padded); later reused as logits[4096]
    float* wts = xs + 128 * 65;      // [128][40]
    float* hs = wts + 128 * 40;      // [40][64] : rows 0-31 policy hidden, 32-39 value hidden (flatten index c*64+sq)
    float* red = hs + 40 * 64;       // [64] scratch
    const int n = n_dev ? *n_dev : n_static;
    const int b = blockIdx.x;
    if (b >= n) return;
    const int t = threadIdx.x;
    {
        const float* src = tower + (size_t)b * 128 * 64;
        for (int i = t; i < 128 * 64; i += 256) xs[(i >> 6) * 65 + (i & 63)] = src[i];
    }
    for (int i = t; i < 128 * 40; i += 256) wts[i] = w40t[i];
    __syncthreads();
    {   // stage 1: 40 outputs per square; thread = (square, group of 10 outputs)
        const int sq = t & 63, og = (t >> 6) * 10;
        float acc[10];
#pragma unroll
        for (int j = 0; j < 10; j++) acc[j] = b40[og + j];
        for (int c = 0; c < 128; c++) {
            const float x = xs[c * 65 + sq];
#pragma unroll
            for (int j = 0; j < 10; j++) acc[j] = fmaf(wts[c * 40 + og + j], x, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < 10; j++) hs[(og + j) * 64 + sq] = fmaxf(acc[j], 0.0f);
    }
    __syncthreads();
    float* logits = xs;  // tower tile no longer needed
    float lmax = -INFINITY;
    {   // stage 2: logits[co*64+sq], thread = (square, 16 output channels)
        const int sq = t & 63, cg = (t >> 6) * 16;
        float acc[16];
#pragma unroll
        for (int j = 0; j < 16; j++) acc[j] = bp2[cg + j];
        for (int k = 0; k < 32; k++) {
            const float x = hs[k * 64 + sq];
#pragma unroll
            for (int j = 0; j < 16; j++) acc[j] = fmaf(__ldg(wp2t + k * 64 + cg + j), x, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < 16; j++) { logits[(cg + j) * 64 + sq] = acc[j]; lmax = fmaxf(lmax, acc[j]); }
    }
    // block max
    for (int d = 16; d; d >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, d));
    if ((t & 31) == 0) red[t >> 5] = lmax;
    __syncthreads();
    float gmax = red[0];
#pragma unroll
    for (int i = 1; i < 8; i++) gmax = fmaxf(gmax, red[i]);
    __syncthreads();
    float lsum = 0.0f;
    for (int i = t; i < 4096; i += 256) {
        float ev = expf(logits[i] - gmax);
        logits[i] = ev;
        lsum += ev;
    }
    for (int d = 16; d; d >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, d);
    if ((t & 31) == 0) red[8 + (t >> 5)] = lsum;
    __syncthreads();
    float gsum = 0.0f;
#pragma unroll
    for (int i = 0; i < 8; i++) gsum += red[8 + i];
    if (policy_out) {
        float* po = policy_out + (size_t)b * 4096;
        for (int i = t; i < 4096; i += 256) po[i] = __fdiv_rn(logits[i], gsum);
    }
    // value head: hidden[t] for t < 64
    if (t < 64) {
        float acc = bl1[t];
        const float* v1 = hs + 32 * 64;  // [8][64] flattened c*64+sq
        for (int i = 0; i < 512; i++) acc = fmaf(v1[i], __ldg(wl1 + i * 64 + t), acc);
        acc = fmaxf(acc, 0.0f) * wl2[t];
        for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if ((t & 31) == 0) red[16 + (t >> 5)] = acc;
    }
    __syncthreads();
    if (t == 0) value_out[b] = tanhf(red[16] + red[17] + bl2[0]);
}

static int launch_heads_f32(az_engine* e, const NetWeights* w, const float* tower, const int* n_dev, int n_static, int grid, float* policy_out,
                            float* value_out) {
    static PerDeviceOnce once;
    if (once.first()) cudaFuncSetAttribute(k_heads_f32, cudaFuncAttributeMaxDynamicSharedMemorySize, HEAD_SMEM);
    if (grid <= 0) return 0;
    k_heads_f32<<<grid, 256, HEAD_SMEM, e->stream>>>(tower, w->f_w40t, w->f_b40, w->f_wp2t, w->f_bp2, w->f_wl1, w->f_bl1,
                                                                  w->f_wl2, w->f_bl2, policy_out, value_out, n_dev, n_static);
    return check_cuda(e, cudaGetLastError(), "k_heads");
}

int net_forward_bf16(az_engine* e, const int* n_dev, int n_static, float* policy_out, float* value_out, const HeadScatter* scatter,
                     const NetBatch* nb) {
    NetWeights* w = e->net;   // the activations, and network 0
    // A multi-network batch (nb, the default configuration only: net_forward_networks) runs the *_nets kernels, which split their
    // CTAs between the two networks.  A network without boards gets no tiles, so when its slot is empty the other network's
    // weights stand in as kernel arguments.
    const NetWeights* wn1 = (e->net1 && e->net1->loaded) ? e->net1 : w;
    const NetWeights* wn0 = w->loaded ? w : wn1;
    if (!wn0->loaded || (!nb && !w->loaded)) return set_err(e, AZ_ERR_NO_WEIGHTS, "az_load_weights has not been called");
    const int grid = e->sm_count & ~1;
    const int tgrid = e->knobs.tower_grid > 0 ? std::min(grid, e->knobs.tower_grid & ~1) : grid;   // CTAs of the tower launch
    const int rel = e->knobs.tc_release_arrive;
    e->n_launches += 1;  // heads; the input convolution and the tower add 1 (one fused launch), 2 or 21 below
    const bool sample = e->prof_every > 0 && (e->prof_counter++ % (uint64_t)e->prof_every) == 0 && e->prof_pending.size() < 4000;
    az_engine::ProfSample ps{nullptr, nullptr, nullptr, nullptr, nullptr, 0};
    if (sample) {
        ps.adv = e->prof_adv_event; e->prof_adv_event = nullptr;
        cudaEventCreate(&ps.in0); cudaEventRecord(ps.in0, e->stream);
    }
    // AZ_TOWER_FUSED: 1 (default) = input convolution + one launch for the 20 tower layers, 2 = the input convolution runs as
    // an extra first layer of that launch (measured: 48 us inside vs 60 us alone per 4096 boards, epilogue-bound either
    // way, so the wave gains 0.2 % -- kept as an option), 0 = 21 launches
    // the input convolution can only run inside the tower launch (mode 2) with the 64-channel plane layout
    const int wide = e->knobs.tower_wide;
    const int fused = (e->knobs.tower_fused >= 2 && (w->in_ch != 64 || wide)) ? 1 : e->knobs.tower_fused;
    int r = 0;
    if (nb) {
        e->n_launches += 1;
        r = tc_conv3x3_nets_launch(e->stream, &w->map_a_in, &wn0->map_w_in, &wn1->map_w_in, wn0->f_b_in, wn1->f_b_in, w->a_buf[0],
                                   nb->counts_dev, nb->base1, grid, (rel ? 32 : 0) | ((e->knobs.tower_l2hint & 8) ? 512 : 0));
        if (r) return set_err(e, AZ_ERR_CUDA, "tc conv (input, networks) launch failed");
    } else if (fused < 2) {
        e->n_launches += 1;
        r = tc_conv3x3_launch(e->stream, &w->map_a_in, &w->map_w_in, w->in_ch, w->f_b_in, nullptr, w->a_buf[0], n_dev, n_static, 1, grid,
                              (rel ? 32 : 0) | ((e->knobs.tower_l2hint & 8) ? 512 : 0) | (e->knobs.input_epi2 ? 1024 : 0));
        if (r) return set_err(e, AZ_ERR_CUDA, "tc conv (input) launch failed");
    }
    if (sample) {
        cudaEventCreate(&ps.a); cudaEventCreate(&ps.b);
        ps.slot = e->prof_slot; e->prof_slot = (e->prof_slot + 1) % 4096;
        cudaEventRecord(ps.a, e->stream);
    }
    int x = 0;  // buffer holding the block input
    if (nb) {
        void* act[3] = {w->a_buf[0], w->a_buf[1], w->a_buf[2]};
        e->n_launches += 1;
        if (sample) e->prof_launches += 1;
        r = tc_tower_nets_launch(e->stream, wn0->d_maps, wn1->d_maps, wn0->f_b_tower, wn1->f_b_tower, act, nb->counts_dev, nb->base1, tgrid,
                                 rel, e->knobs.tower_l2hint);
        if (r) return set_err(e, AZ_ERR_CUDA, "tower (networks) launch failed");
    } else if (fused) {
        void* act[3] = {w->a_buf[0], w->a_buf[1], w->a_buf[2]};
        // The tower runs over consecutive board ranges whose two activation buffers (block input/output in place, conv1
        // output) stay resident in the 126 MB L2: a range of 2048 boards is 2 x 33.5 MB, and 512 tiles on 74 CTA pairs
        // are 7 rounds, the same 98.8 % fill as the whole batch.  At 4096 boards two launches take 1148 us against
        // 1250 us for one launch whose 134 MB stream through HBM in every layer (and the clocks under the power cap
        // are higher).  AZ_TOWER_SPLIT overrides the number of ranges.
        const int split = e->knobs.tower_split;
        const int cap_tiles = ((n_dev ? w->max_boards : n_static) + 3) / 4;
        const int pairs = tgrid / 2;
        int n_ranges = split > 0 ? split : (cap_tiles + 7 * pairs - 1) / (7 * pairs);   // at most 7 rounds (2072 boards) per range
        if (split == 0 && cap_tiles < 6 * pairs * n_ranges) n_ranges = std::max(1, cap_tiles / (6 * pairs));  // >= 6 tiles per pair (lazy publication)
        const int per = (cap_tiles + n_ranges - 1) / n_ranges;
        // One launch walks all ranges (all 20 layers of a range, then the next range: the weight pipeline simply continues),
        // which saves a launch fill/drain per extra range; AZ_TOWER_INKERNEL=0 launches once per range instead.
        const int inkernel = e->knobs.tower_inkernel;
        for (int lo = 0; lo < cap_tiles; lo += inkernel ? cap_tiles : per) {
            e->n_launches += 1;
            if (sample) e->prof_launches += 1;
            r = inkernel ? tc_tower_launch(e->stream, w->d_maps, w->f_b_tower, act, n_dev, n_static, 20, fused >= 2, tgrid, 0, 0x7FFFFFFF, per, rel, wide, e->knobs.tower_l2hint)
                         : tc_tower_launch(e->stream, w->d_maps, w->f_b_tower, act, n_dev, n_static, 20, fused >= 2, tgrid, lo, lo + per, 0, rel, wide, e->knobs.tower_l2hint);
            if (r) return set_err(e, AZ_ERR_CUDA, "tower launch failed");
        }
        x = 0;  // the fused tower works in place: block input and block output share a_buf[0], a_buf[1] holds conv1's output
    }
    for (int blk = 0; blk < (fused || nb ? 0 : 10); blk++) {
        e->n_launches += 2;
        if (sample) e->prof_launches += 2;
        const int y = (x + 1) % 3, z = (x + 2) % 3;
        r = tc_conv3x3_launch(e->stream, &w->map_a[x], &w->map_w_tower[2 * blk], 128, w->f_b_tower + (2 * blk) * 128, nullptr, w->a_buf[y],
                              n_dev, n_static, 1, grid, rel ? 32 : 0);
        if (r) return set_err(e, AZ_ERR_CUDA, "tc conv launch failed");
        r = tc_conv3x3_launch(e->stream, &w->map_a[y], &w->map_w_tower[2 * blk + 1], 128, w->f_b_tower + (2 * blk + 1) * 128, w->a_buf[x],
                              w->a_buf[z], n_dev, n_static, 1, grid, rel ? 32 : 0);
        if (r) return set_err(e, AZ_ERR_CUDA, "tc conv launch failed");
        x = z;
    }
    if (sample) cudaEventRecord(ps.b, e->stream);
    const int hr = nb ? launch_heads_tc_nets(e, wn0, wn1, &w->map_rows[x], nb->counts_dev, nb->base1, nb->cap, policy_out, value_out, scatter)
                 : e->knobs.heads_tc ? launch_heads_tc(e, &w->map_rows[x], n_dev, n_static, policy_out, value_out, scatter)
                                     : launch_heads_mma(e, w->a_buf[x], n_dev, n_static, policy_out, value_out, scatter);
    if (sample) {
        cudaEventCreate(&ps.h1); cudaEventRecord(ps.h1, e->stream);
        // the batch size of this wave, copied after the last bracketed phase so that the copy is not timed as part of one
        if (n_dev) cudaMemcpyAsync(&e->prof_counts_host[ps.slot], n_dev, sizeof(int), cudaMemcpyDeviceToHost, e->stream);
        else e->prof_counts_host[ps.slot] = n_static;
        e->prof_pending.push_back(ps);
    }
    return hr;
}

int net_forward_fp32(az_engine* e, const float* planes, const int* n_dev, int n_static, float* policy_out, float* value_out,
                     const NetWeights* wts) {
    NetWeights* w = e->net;
    if (!wts) wts = w;
    if (!wts->loaded) return set_err(e, AZ_ERR_NO_WEIGHTS, "az_load_weights has not been called");
    for (int i = 0; i < 3; i++)
        if (!w->g_buf[i]) AZ_CUDA(e, cudaMalloc(&w->g_buf[i], (size_t)w->max_boards * 128 * 64 * sizeof(float)));
    static PerDeviceOnce once;
    if (once.first()) cudaFuncSetAttribute(k_conv3x3_f32<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 64 * 4);
    const int grid = n_dev ? w->max_boards : n_static;
    if (grid <= 0) return 0;
    e->n_launches += 22;
    k_conv3x3_f32<19><<<grid, 256, 19 * 64 * 4, e->stream>>>(planes, wts->f_w_in, wts->f_b_in, nullptr, w->g_buf[0], n_dev, n_static, 1);
    int x = 0;
    for (int blk = 0; blk < 10; blk++) {
        const int y = (x + 1) % 3, z = (x + 2) % 3;
        k_conv3x3_f32<128><<<grid, 256, 128 * 64 * 4, e->stream>>>(w->g_buf[x], wts->f_w_tower + (size_t)(2 * blk) * 128 * 128 * 9,
                                                                  wts->f_b_tower + (2 * blk) * 128, nullptr, w->g_buf[y], n_dev, n_static, 1);
        k_conv3x3_f32<128><<<grid, 256, 128 * 64 * 4, e->stream>>>(w->g_buf[y], wts->f_w_tower + (size_t)(2 * blk + 1) * 128 * 128 * 9,
                                                                  wts->f_b_tower + (2 * blk + 1) * 128, w->g_buf[x], w->g_buf[z], n_dev,
                                                                  n_static, 1);
        x = z;
    }
    AZ_CUDA(e, cudaGetLastError());
    return launch_heads_f32(e, wts, w->g_buf[x], n_dev, n_static, grid, policy_out, value_out);
}

int net_forward_networks(az_engine* e, const NetBatch& nb, const float* planes_f32, float* policy_out, float* value_out,
                         const HeadScatter* scatter) {
    if (e->cfg.precision == 1) {   // the parity path: one network after the other over its range
        for (int s = 0; s < AZ_MAX_NETWORKS; s++) {
            const NetWeights* ws = net_slot(e, s);
            if (!ws || !ws->loaded) continue;   // callers route no board to a network that was never loaded
            const int base = s ? nb.base1 : 0;
            const int r = net_forward_fp32(e, planes_f32 + (size_t)base * AZ_NUM_PLANES * 64, nb.counts_dev + s, 0,
                                           policy_out ? policy_out + (size_t)base * AZ_ACTION_SPACE : nullptr, value_out + base, ws);
            if (r) return r;
        }
        return 0;
    }
    const int r = net_networks_supported(e);
    if (r) return r;
    return net_forward_bf16(e, nullptr, nb.cap, policy_out, value_out, scatter, &nb);
}

int net_networks_supported(az_engine* e) {
    const az_engine::Knobs& k = e->knobs;
    if (e->cfg.precision != 1 && (k.tower_fused != 1 || k.tower_wide != 2 || k.tower_inkernel != 1 || k.tower_split != 0 || k.input_k32 != 1 ||
                                  k.input_epi2 != 0 || k.heads_tc != 1))
        return set_err(e, AZ_ERR_STATE, "a multi-network forward needs the default AZ_TOWER_*, AZ_INPUT_* and AZ_HEADS_TC configuration");
    return AZ_OK;
}

}  // namespace azb

using namespace azb;

extern "C" {

const char* az_weight_name(int i) {
    static std::string names[AZ_NUM_WEIGHT_ARRAYS];
    if (i < 0 || i >= AZ_NUM_WEIGHT_ARRAYS) return "";
    if (names[i].empty()) names[i] = weight_name(i);
    return names[i].c_str();
}
int64_t az_weight_size(int i) { return (i < 0 || i >= AZ_NUM_WEIGHT_ARRAYS) ? 0 : weight_size(i); }

int az_load_weights(az_engine* e, const float* const* arrays, int n_arrays) {
    if (!e || !arrays) return AZ_ERR_INVALID_ARGUMENT;
    if (n_arrays != AZ_NUM_WEIGHT_ARRAYS) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "expected AZ_NUM_WEIGHT_ARRAYS tensors");
    for (int i = 0; i < n_arrays; i++) if (!arrays[i]) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null weight tensor");
    cudaSetDevice(e->cfg.device);
    return load_from_host(e, e->net, arrays);
}

int az_load_network(az_engine* e, int network, const float* const* arrays, int n_arrays) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (network < 0 || network >= AZ_MAX_NETWORKS) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "network must be in [0, AZ_MAX_NETWORKS)");
    if (network == 0) return az_load_weights(e, arrays, n_arrays);
    if (!arrays) return AZ_ERR_INVALID_ARGUMENT;
    if (n_arrays != AZ_NUM_WEIGHT_ARRAYS) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "expected AZ_NUM_WEIGHT_ARRAYS tensors");
    for (int i = 0; i < n_arrays; i++) if (!arrays[i]) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null weight tensor");
    cudaSetDevice(e->cfg.device);
    if (!e->net1) {
        const int r = create_slot1(e);
        if (r) return r;
    }
    return load_from_host(e, e->net1, arrays);
}

int az_load_weights_dev(az_engine* e, const float* const* arrays_dev, int n_arrays) {
    if (!e || !arrays_dev) return AZ_ERR_INVALID_ARGUMENT;
    if (n_arrays != AZ_NUM_WEIGHT_ARRAYS) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "expected AZ_NUM_WEIGHT_ARRAYS tensors");
    cudaSetDevice(e->cfg.device);
    std::vector<std::vector<float>> host(n_arrays);
    std::vector<const float*> ptrs(n_arrays);
    for (int i = 0; i < n_arrays; i++) {
        host[i].resize((size_t)weight_size(i));
        AZ_CUDA(e, cudaMemcpy(host[i].data(), arrays_dev[i], host[i].size() * 4, cudaMemcpyDeviceToHost));
        ptrs[i] = host[i].data();
    }
    return load_from_host(e, e->net, ptrs.data());
}

static int forward_common(az_engine* e, int n, float* policy_out, float* value_out) {
    AZ_CUDA(e, cudaMemcpyAsync(policy_out, e->d_policy, (size_t)n * AZ_ACTION_SPACE * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(value_out, e->d_value, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

int az_forward_planes(az_engine* e, int n, const float* planes, float* policy_out, float* value_out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (n < 0 || n > e->max_batch) return set_err(e, AZ_ERR_CAPACITY, "batch larger than az_config.max_batch");
    if (n == 0) return AZ_OK;
    if (!planes || !policy_out || !value_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    cudaSetDevice(e->cfg.device);
    AZ_CUDA(e, cudaMemcpyAsync(e->d_planes, planes, (size_t)n * AZ_NUM_PLANES * 64 * 4, cudaMemcpyHostToDevice, e->stream));
    int r;
    if (e->cfg.precision == 1) {
        r = net_forward_fp32(e, e->d_planes, nullptr, n, e->d_policy, e->d_value);
    } else {
        launch_planes_to_bf16(e->stream, e->d_planes, e->net->a_in, n, e->net->in_ch);
        r = net_forward_bf16(e, nullptr, n, e->d_policy, e->d_value);
    }
    if (r) return r;
    return forward_common(e, n, policy_out, value_out);
}

int az_forward(az_engine* e, int n, const az_position* pos, float* policy_out, float* value_out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (n < 0 || n > e->max_batch) return set_err(e, AZ_ERR_CAPACITY, "batch larger than az_config.max_batch");
    if (n == 0) return AZ_OK;
    if (!pos || !policy_out || !value_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    cudaSetDevice(e->cfg.device);
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, pos, (size_t)n * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    int r;
    if (e->cfg.precision == 1) {
        launch_encode_f32(e->stream, e->d_wire, e->d_planes, n);
        r = net_forward_fp32(e, e->d_planes, nullptr, n, e->d_policy, e->d_value);
    } else {
        launch_encode_bf16_wire(e->stream, e->d_wire, e->net->a_in, n, e->net->in_ch);
        r = net_forward_bf16(e, nullptr, n, e->d_policy, e->d_value);
    }
    if (r) return r;
    return forward_common(e, n, policy_out, value_out);
}

int az_forward_networks(az_engine* e, int n, const az_position* pos, const uint8_t* network, float* policy_out, float* value_out) {
    if (!e) return AZ_ERR_INVALID_ARGUMENT;
    if (n < 0 || n > e->max_batch) return set_err(e, AZ_ERR_CAPACITY, "batch larger than az_config.max_batch");
    if (n == 0) return AZ_OK;
    if (!pos || !network || !policy_out || !value_out) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "null buffer");
    int count[AZ_MAX_NETWORKS] = {0, 0};
    for (int i = 0; i < n; i++) {
        if (network[i] >= AZ_MAX_NETWORKS) return set_err(e, AZ_ERR_INVALID_ARGUMENT, "network id must be < AZ_MAX_NETWORKS");
        count[network[i]]++;
    }
    for (int s = 0; s < AZ_MAX_NETWORKS; s++) {
        const NetWeights* w = net_slot(e, s);
        if (count[s] && (!w || !w->loaded)) return set_err(e, AZ_ERR_NO_WEIGHTS, "a board names a network that has not been loaded");
    }
    // network ranges: network 0 at board 0, network 1 at the next multiple of 4 (a tile of the convolutions never mixes networks)
    const int base1 = (count[0] + 3) & ~3;
    if (base1 + ((count[1] + 3) & ~3) > e->max_batch) return set_err(e, AZ_ERR_CAPACITY, "network ranges exceed az_config.max_batch");
    const int span = base1 + count[1];
    std::vector<az_position> staged((size_t)span, pos[0]);   // the padding between the ranges is never evaluated
    std::vector<int> slot(n);
    int next[AZ_MAX_NETWORKS] = {0, base1};
    for (int i = 0; i < n; i++) { slot[i] = next[network[i]]++; staged[slot[i]] = pos[i]; }
    cudaSetDevice(e->cfg.device);
    if (!e->d_net_counts) {
        AZ_CUDA(e, cudaMalloc(&e->d_net_counts, AZ_MAX_NETWORKS * sizeof(int)));
        AZ_CUDA(e, cudaMalloc(&e->d_net_slot, (size_t)e->max_batch * sizeof(int)));
        AZ_CUDA(e, cudaMalloc(&e->d_net_value, (size_t)e->max_batch * sizeof(float)));
    }
    if (!e->d_scores) AZ_CUDA(e, cudaMalloc(&e->d_scores, (size_t)e->max_batch * AZ_ACTION_SPACE * 4));
    AZ_CUDA(e, cudaMemcpyAsync(e->d_net_counts, count, sizeof count, cudaMemcpyHostToDevice, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(e->d_net_slot, slot.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(e->d_wire, staged.data(), (size_t)span * sizeof(az_position), cudaMemcpyHostToDevice, e->stream));
    if (e->cfg.precision == 1) launch_encode_f32(e->stream, e->d_wire, e->d_planes, span);
    else launch_encode_bf16_wire(e->stream, e->d_wire, e->net->a_in, span, e->net->in_ch);
    const int r = net_forward_networks(e, NetBatch{e->d_net_counts, base1, span}, e->d_planes, e->d_policy, e->d_value);
    if (r) return r;
    // back to the caller's order (the scores export buffer holds the gathered policy rows)
    e->n_launches++;
    k_gather_rows<<<n, 256, 0, e->stream>>>(e->d_policy, e->d_value, e->d_net_slot, e->d_scores, e->d_net_value);
    AZ_CUDA(e, cudaGetLastError());
    AZ_CUDA(e, cudaMemcpyAsync(policy_out, e->d_scores, (size_t)n * AZ_ACTION_SPACE * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaMemcpyAsync(value_out, e->d_net_value, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    AZ_CUDA(e, cudaStreamSynchronize(e->stream));
    return AZ_OK;
}

}  // extern "C"
