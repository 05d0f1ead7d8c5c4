// Diagnostic entry points: run one encoder kernel on host data (kernel-level numerics tests).
#include <vector>

#include "attention.cuh"
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

using namespace mb;

namespace {

struct Scratch {
    std::vector<void*> ptrs;
    cudaStream_t s = nullptr;
    ~Scratch() {
        for (void* p : ptrs) cudaFree(p);
        if (s) cudaStreamDestroy(s);
    }
    template <class T>
    T* alloc(size_t n) {
        void* p = nullptr;
        MB_CUDA(cudaMalloc(&p, std::max<size_t>(n * sizeof(T), 16)));
        ptrs.push_back(p);
        return reinterpret_cast<T*>(p);
    }
    template <class T>
    T* upload(const T* h, size_t n) {
        T* d = alloc<T>(n);
        MB_CUDA(cudaMemcpy(d, h, n * sizeof(T), cudaMemcpyHostToDevice));
        return d;
    }
    __nv_bfloat16* upload_bf16(const float* h, size_t n) {
        float* f = upload(h, n);
        __nv_bfloat16* b = alloc<__nv_bfloat16>(n);
        kernels::f32_to_bf16(f, b, (long long)n, s);
        return b;
    }
};

__global__ void bf16_to_f32_kernel(const __nv_bfloat16* src, float* dst, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = __bfloat162float(src[i]);
}

// pseudo-random bf16 values in [-1, 1) (kernel timing probes: no 200 MB host upload)
__global__ void fill_bf16_kernel(__nv_bfloat16* dst, long long n, uint32_t seed) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t x = (uint32_t)i * 2654435761u + seed;
    x ^= x >> 16;
    x *= 0x85ebca6bu;
    x ^= x >> 13;
    dst[i] = __float2bfloat16_rn((float)(x & 0xFFFF) / 32768.0f - 1.0f);
}

void require_device(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        fail(B200_ERR_NO_DEVICE, "CUDA device %d not available (marqo_b200 has no CPU fallback)", device);
    }
}

}  // namespace

extern "C" {

int b200_debug_patch_embed(int device, const uint8_t* hwc, int n, int S, int patch, const float* conv_w, int N,
                           const float* mean3, const float* std3, const float* pos, int use_gather, float* out) {
    return guarded([&] {
        MB_CHECK_ARG(hwc && conv_w && mean3 && std3 && out, "NULL buffer");
        MB_CHECK_ARG(n > 0 && S > 0 && patch > 0 && S % patch == 0 && N > 0 && N % 32 == 0, "bad shape");
        require_device(device);
        DeviceGuard g(device);
        Scratch sc;
        MB_CUDA(cudaStreamCreate(&sc.s));
        const int G = (S / patch) * (S / patch), K = 3 * patch * patch;
        uint8_t* dImg = sc.upload(hwc, (size_t)n * S * S * 3);
        float* dW = sc.upload(conv_w, (size_t)N * K);
        float* dOut = sc.alloc<float>((size_t)n * (G + 1) * N);
        MB_CUDA(cudaMemsetAsync(dOut, 0, (size_t)n * (G + 1) * N * 4, sc.s));
        gemm::Epilogue ep;
        ep.out = dOut;
        ep.ldo = N;
        ep.out_fp32 = 1;
        ep.remap_group = G;                                   // token row b * (G + 1) + 1 + i, as the ViT forward does
        ep.rowbias = pos ? sc.upload(pos, (size_t)(G + 1) * N) : nullptr;
        if (!pos) ep.rowbias = nullptr;
        int sms = sm_count(device);
        if (use_gather) {
            MB_CHECK_ARG(gemm::patch_gather_supported(S, patch), "the gather GEMM does not support image %d / patch %d", S,
                         patch);
            __nv_bfloat16* dWg = sc.alloc<__nv_bfloat16>((size_t)N * gemm::patch_gather_k(patch));
            kernels::patch_weight_rows(dW, N, patch, gemm::patch_gather_kbpd(patch), dWg, sc.s);
            gemm::PatchGather pg;
            pg.img = dImg;
            pg.n = n;
            pg.S = S;
            pg.patch = patch;
            for (int i = 0; i < 3; ++i) {
                pg.mean[i] = mean3[i];
                pg.std[i] = std3[i];
            }
            gemm::launch_patch_embed(pg, dWg, N, ep, sms, sc.s);
        } else {
            const int kpad = (int)round_up((size_t)K, 64);
            __nv_bfloat16* dWp = sc.alloc<__nv_bfloat16>((size_t)N * kpad);
            kernels::pad_rows_to_bf16(dW, N, K, kpad, dWp, sc.s);
            __nv_bfloat16* dP = sc.alloc<__nv_bfloat16>((size_t)n * G * kpad);
            kernels::im2col_u8(dImg, n, S, patch, kpad, mean3, std3, dP, sc.s);
            gemm::launch(dP, kpad, dWp, n * G, N, kpad, ep, sms, sc.s);
        }
        MB_CUDA(cudaMemcpyAsync(out, dOut, (size_t)n * (G + 1) * N * 4, cudaMemcpyDeviceToHost, sc.s));
        MB_CUDA(cudaStreamSynchronize(sc.s));
    });
}

int b200_debug_gemm(int device, const float* A, const float* W, const float* bias, const float* residual, int M, int N,
                    int K, int act, int out_bf16, int in_place, float* out) {
    return guarded([&] {
        MB_CHECK_ARG(A && W && out, "NULL buffer");
        MB_CHECK_ARG(M > 0 && N > 0 && K > 0, "M, N, K must be positive");
        MB_CHECK_ARG(!in_place || (residual && !out_bf16), "in_place needs a residual and fp32 output");
        require_device(device);
        DeviceGuard g(device);
        Scratch sc;
        MB_CUDA(cudaStreamCreate(&sc.s));
        __nv_bfloat16* dA = sc.upload_bf16(A, (size_t)M * K);
        __nv_bfloat16* dW = sc.upload_bf16(W, (size_t)N * K);
        // in place: the residual is uploaded into the output buffer, as out_proj / fc2 add onto the residual stream
        float* dOut = in_place ? sc.upload(residual, (size_t)M * N) : sc.alloc<float>((size_t)M * N);
        gemm::Epilogue ep;
        ep.bias = bias ? sc.upload(bias, (size_t)N) : nullptr;
        ep.residual = in_place ? dOut : residual ? sc.upload(residual, (size_t)M * N) : nullptr;
        ep.ldr = N;
        ep.act = act;
        ep.ldo = N;
        __nv_bfloat16* dOutB = nullptr;
        if (out_bf16) {
            dOutB = sc.alloc<__nv_bfloat16>((size_t)M * N);
            ep.out = dOutB;
            ep.out_fp32 = 0;
        } else {
            ep.out = dOut;
            ep.out_fp32 = 1;
        }
        gemm::launch(dA, K, dW, M, N, K, ep, sm_count(device), sc.s);
        if (out_bf16) {
            const long long n = (long long)M * N;
            bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, sc.s>>>(dOutB, dOut, n);
        }
        MB_CUDA(cudaGetLastError());
        MB_CUDA(cudaStreamSynchronize(sc.s));
        MB_CUDA(cudaMemcpy(out, dOut, (size_t)M * N * 4, cudaMemcpyDeviceToHost));
    });
}

int b200_debug_attention(int device, const float* qkv, int B, int S, int W, int H, int mask, const int32_t* kv_len,
                         float* out) {
    return guarded([&] {
        MB_CHECK_ARG(qkv && out, "NULL buffer");
        MB_CHECK_ARG(B > 0 && S > 0 && W > 0 && H > 0, "B, S, W, H must be positive");
        require_device(device);
        DeviceGuard g(device);
        Scratch sc;
        MB_CUDA(cudaStreamCreate(&sc.s));
        const size_t M = (size_t)B * S;
        __nv_bfloat16* dq = sc.upload_bf16(qkv, M * 3 * W);
        __nv_bfloat16* dO = sc.alloc<__nv_bfloat16>(M * W);
        float* dOut = sc.alloc<float>(M * W);
        const int32_t* dlen = kv_len ? sc.upload(kv_len, (size_t)B) : nullptr;
        attention::launch(dq, dO, B, S, W, H, mask, dlen, nullptr, sc.s);
        const long long n = (long long)M * W;
        bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, sc.s>>>(dO, dOut, n);
        MB_CUDA(cudaGetLastError());
        MB_CUDA(cudaStreamSynchronize(sc.s));
        MB_CUDA(cudaMemcpy(out, dOut, M * W * 4, cudaMemcpyDeviceToHost));
    });
}

int b200_debug_attention_relbias(int device, const float* qkv, int B, int S, int W, int H, int mask,
                                 const int32_t* kv_len, const float* rel_bias, float* out) {
    return guarded([&] {
        MB_CHECK_ARG(qkv && rel_bias && out, "NULL buffer");
        MB_CHECK_ARG(B > 0 && S > 0 && W > 0 && H > 0, "B, S, W, H must be positive");
        MB_CHECK_ARG(mask == attention::MASK_NONE || mask == attention::MASK_KEYLEN, "mask must be 0 (none) or 2 (key length)");
        require_device(device);
        DeviceGuard g(device);
        Scratch sc;
        MB_CUDA(cudaStreamCreate(&sc.s));
        const size_t M = (size_t)B * S;
        std::vector<float> folded((size_t)H * attention::REL_T);
        attention::fold_relative_bias(rel_bias, H, S - 1, folded.data());
        const float* dbias = sc.upload(folded.data(), folded.size());
        __nv_bfloat16* dq = sc.upload_bf16(qkv, M * 3 * W);
        __nv_bfloat16* dO = sc.alloc<__nv_bfloat16>(M * W);
        float* dOut = sc.alloc<float>(M * W);
        const int32_t* dlen = kv_len ? sc.upload(kv_len, (size_t)B) : nullptr;
        attention::launch(dq, dO, B, S, W, H, mask, dlen, dbias, sc.s);
        const long long n = (long long)M * W;
        bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, sc.s>>>(dO, dOut, n);
        MB_CUDA(cudaGetLastError());
        MB_CUDA(cudaStreamSynchronize(sc.s));
        MB_CUDA(cudaMemcpy(out, dOut, M * W * 4, cudaMemcpyDeviceToHost));
    });
}

int b200_debug_relative_position_buckets(int max_distance, int32_t* out) {
    return guarded([&] {
        MB_CHECK_ARG(out != nullptr, "NULL buffer");
        MB_CHECK_ARG(max_distance >= 0, "max_distance must be >= 0");
        for (int d = -max_distance; d <= max_distance; ++d) out[d + max_distance] = attention::relative_position_bucket(d);
    });
}

int b200_debug_attention_time(int device, int B, int S, int W, int H, int mask, int iters, float* out_ms) {
    return guarded([&] {
        MB_CHECK_ARG(out_ms != nullptr, "NULL buffer");
        MB_CHECK_ARG(B > 0 && S > 0 && W > 0 && H > 0 && iters > 0, "B, S, W, H, iters must be positive");
        require_device(device);
        DeviceGuard g(device);
        Scratch sc;
        MB_CUDA(cudaStreamCreate(&sc.s));
        const size_t M = (size_t)B * S;
        __nv_bfloat16* dq = sc.alloc<__nv_bfloat16>(M * 3 * W);
        __nv_bfloat16* dO = sc.alloc<__nv_bfloat16>(M * W);
        const long long n = (long long)(M * 3 * W);
        fill_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, sc.s>>>(dq, n, 12345u);
        MB_CUDA(cudaGetLastError());
        std::vector<int32_t> lens((size_t)B, S);
        const int32_t* dlen = mask == attention::MASK_KEYLEN ? sc.upload(lens.data(), (size_t)B) : nullptr;
        cudaEvent_t e0, e1;
        MB_CUDA(cudaEventCreate(&e0));
        MB_CUDA(cudaEventCreate(&e1));
        for (int i = 0; i < 3; ++i) attention::launch(dq, dO, B, S, W, H, mask, dlen, nullptr, sc.s);   // warm-up
        MB_CUDA(cudaEventRecord(e0, sc.s));
        for (int i = 0; i < iters; ++i) attention::launch(dq, dO, B, S, W, H, mask, dlen, nullptr, sc.s);
        MB_CUDA(cudaEventRecord(e1, sc.s));
        MB_CUDA(cudaStreamSynchronize(sc.s));
        float ms = 0.f;
        MB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        *out_ms = ms / (float)iters;
    });
}

int b200_debug_layernorm(int device, const float* x, const float* gamma, const float* beta, float eps, int rows, int w,
                         float* out) {
    return guarded([&] {
        MB_CHECK_ARG(x && gamma && beta && out, "NULL buffer");
        require_device(device);
        DeviceGuard g(device);
        Scratch sc;
        MB_CUDA(cudaStreamCreate(&sc.s));
        float* dx = sc.upload(x, (size_t)rows * w);
        float* dg = sc.upload(gamma, (size_t)w);
        float* db = sc.upload(beta, (size_t)w);
        float* dout = sc.alloc<float>((size_t)rows * w);
        kernels::layernorm(dx, w, dg, db, eps, rows, w, dout, nullptr, sc.s);
        MB_CUDA(cudaStreamSynchronize(sc.s));
        MB_CUDA(cudaMemcpy(out, dout, (size_t)rows * w * 4, cudaMemcpyDeviceToHost));
    });
}

int b200_debug_resize(int device, const uint8_t* hwc, int n, int h, int w, int S, uint8_t* out) {
    return guarded([&] {
        MB_CHECK_ARG(hwc && out, "NULL buffer");
        MB_CHECK_ARG(n > 0 && h > 0 && w > 0 && S > 0, "n, h, w, S must be positive");
        require_device(device);
        DeviceGuard g(device);
        Scratch sc;
        MB_CUDA(cudaStreamCreate(&sc.s));
        uint8_t* din = sc.upload(hwc, (size_t)n * h * w * 3);
        uint8_t* dout = sc.alloc<uint8_t>((size_t)n * S * S * 3);
        kernels::resize_crop_u8(din, n, h, w, S, dout, sc.s);
        MB_CUDA(cudaStreamSynchronize(sc.s));
        MB_CUDA(cudaMemcpy(out, dout, (size_t)n * S * S * 3, cudaMemcpyDeviceToHost));
    });
}

}  // extern "C"
