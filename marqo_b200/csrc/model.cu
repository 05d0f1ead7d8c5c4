// Encoder runtime: CLIP ViT image tower, CLIP text tower, BERT (e5), MPNet (all-mpnet-base-v2) — SURVEY §8 a2-a5.
//
// What the reference calls (third-party, restated in oracle/encoders.py):
//   OPEN_CLIP.encode_image / encode_text   src/marqo/core/inference/embedding_models/open_clip_model.py:249-286
//   HuggingFaceModel.encode                src/marqo/core/inference/embedding_models/hugging_face_model.py:172-214
//
// Data layout in HBM (per model handle):
//   weights   bf16 [out, in] for every Linear (tcgen05 B operand, K-major), fp32 for LayerNorm / biases /
//             embeddings / projections
//   x         fp32 [tokens, width]   residual stream (kept fp32 end to end)
//   h         bf16 [tokens, width]   LayerNorm output = GEMM A operand
//   qkv       bf16 [tokens, 3*width] fused QKV projection
//   o         bf16 [tokens, width]   attention output
//   u         bf16 [tokens, mlp]     MLP hidden
//   patches   bf16 [images * grid^2, kpad]  normalised im2col of the uint8 input (ToTensor + Normalize fused)
// Every Linear is the tcgen05 GEMM of gemm.cu with bias / activation / residual-add fused into its epilogue.
#include <algorithm>
#include <cstdlib>
#include <map>
#include <tuple>
#include <mutex>
#include <string>
#include <vector>

#include "attention.cuh"
#include "common.cuh"
#include "gemm.cuh"
#include "kernels.cuh"

using namespace mb;

namespace {

struct Buf {
    void* p = nullptr;
    size_t bytes = 0;
};

struct LayerW {
    const float *ln1_w = nullptr, *ln1_b = nullptr, *ln2_w = nullptr, *ln2_b = nullptr;
    const float *b_qkv = nullptr, *b_o = nullptr, *b_fc = nullptr, *b_proj = nullptr;
    const __nv_bfloat16 *w_qkv = nullptr, *w_o = nullptr, *w_fc = nullptr, *w_proj = nullptr;
};

struct TowerW {
    b200_tower_desc d{};
    bool present = false;
    std::vector<LayerW> layers;
    // vision
    const __nv_bfloat16* conv_w = nullptr;  // [width, kpad]
    const __nv_bfloat16* conv_wg = nullptr; // [width, gemm::patch_gather_k(patch)]: gather GEMM order, or NULL if unsupported
    int kpad = 0, grid = 0, tokens = 0;
    const float *cls = nullptr, *pos = nullptr, *ln_pre_w = nullptr, *ln_pre_b = nullptr;
    // final LN (ln_post / ln_final) and projection [width, embed]
    const float *ln_out_w = nullptr, *ln_out_b = nullptr, *proj = nullptr;
    // text / bert embeddings
    const float *tok = nullptr, *type0 = nullptr, *emb_ln_w = nullptr, *emb_ln_b = nullptr;
    int max_pos = 0;
    // MPNet: relative-position bias folded to the attention kernels' table [heads, attention::REL_T] (log2 units)
    const float* rel_bias = nullptr;
};

}  // namespace

struct b200_model {
    int device = 0;
    int sms = 0;
    b200_model_desc desc{};
    bool finalized = false;
    std::map<std::string, Buf> raw;   // uploaded fp32 parameters by checkpoint name
    std::vector<void*> owned;         // derived device buffers
    TowerW vision, text;
    // workspaces (sized for max_tokens tokens)
    long long max_tokens = 0;
    float* x = nullptr;
    __nv_bfloat16 *h = nullptr, *qkv = nullptr, *o = nullptr, *u = nullptr, *patches = nullptr;
    int32_t *aux = nullptr;           // [max_batch] eot index / kv_len
    float* out_dev = nullptr;         // [max_batch, embed]
    float* pooled = nullptr;          // [max_batch, width] LayerNorm-ed pooled rows (CLIP heads)
    void* in_dev = nullptr;           // staging for host inputs
    size_t in_dev_bytes = 0;
    uint8_t* resized = nullptr;       // [max_batch, S, S, 3]
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;  // created by the handle; `stream` may be replaced by a caller's stream
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timing_valid = false;
    int last_launches = 0;
    // optional per-kernel-class device timing (bench.py's roofline numerator)
    bool profiling = false;
    std::vector<cudaEvent_t> prof_ev;  // pairs
    std::vector<int> prof_cls;         // 0 = gemm, 1 = attention
    int prof_n = 0;
    // CUDA graphs of small (launch-bound) forward passes, keyed by everything the captured launches depend on
    struct GraphKey {
        int kind, n, S, normalize;
        const void *in0, *in1, *out;
        bool operator<(const GraphKey& o) const {
            return std::tie(kind, n, S, normalize, in0, in1, out) < std::tie(o.kind, o.n, o.S, o.normalize, o.in0, o.in1, o.out);
        }
    };
    struct GraphEntry {
        cudaGraphExec_t exec = nullptr;   // null: seen once (ran eagerly), captured on the next use
        int launches = 0;
    };
    std::map<GraphKey, GraphEntry> graphs;
    bool external_stream = false;
    std::mutex mu;
};

namespace {

void dev_alloc(void** p, size_t bytes) {
    cudaError_t e = cudaMalloc(p, std::max<size_t>(bytes, 16));
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        fail(B200_ERR_OOM, "cudaMalloc(%zu bytes) failed: out of device memory", bytes);
    }
    MB_CUDA(e);
}

void model_free(b200_model* m) {
    if (!m) return;
    cudaSetDevice(m->device);
    for (auto& kv : m->raw) cudaFree(kv.second.p);
    for (void* p : m->owned) cudaFree(p);
    cudaFree(m->x);
    cudaFree(m->h);
    cudaFree(m->qkv);
    cudaFree(m->o);
    cudaFree(m->u);
    cudaFree(m->patches);
    cudaFree(m->aux);
    cudaFree(m->out_dev);
    cudaFree(m->pooled);
    cudaFree(m->in_dev);
    cudaFree(m->resized);
    if (m->ev0) cudaEventDestroy(m->ev0);
    if (m->ev1) cudaEventDestroy(m->ev1);
    for (cudaEvent_t e : m->prof_ev) cudaEventDestroy(e);
    for (auto& kv : m->graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    if (m->own_stream) cudaStreamDestroy(m->own_stream);
    delete m;
}

void check_tower(const b200_tower_desc& t, const char* name) {
    MB_CHECK_ARG(t.width > 0 && t.width % 128 == 0 && t.width <= 1024, "%s.width %d must be a multiple of 128, <= 1024",
                 name, t.width);
    MB_CHECK_ARG(t.layers > 0, "%s.layers must be positive", name);
    MB_CHECK_ARG(t.heads > 0 && t.width == t.heads * 64, "%s: head_dim must be 64 (width %d, heads %d)", name, t.width,
                 t.heads);
    MB_CHECK_ARG(t.mlp > 0 && t.mlp % 64 == 0, "%s.mlp %d must be a multiple of 64", name, t.mlp);
}

const float* param(b200_model* m, const std::string& name, long long numel) {
    auto it = m->raw.find(name);
    if (it == m->raw.end()) fail(B200_ERR_MISSING_WEIGHT, "missing parameter '%s'", name.c_str());
    if ((long long)(it->second.bytes / sizeof(float)) != numel)
        fail(B200_ERR_INVALID_ARG, "parameter '%s' has %zu elements, expected %lld", name.c_str(),
             it->second.bytes / sizeof(float), numel);
    return reinterpret_cast<const float*>(it->second.p);
}

// fp32 parameter -> owned bf16 copy; the fp32 original is released.
const __nv_bfloat16* to_bf16(b200_model* m, const std::string& name, long long numel) {
    const float* src = param(m, name, numel);
    __nv_bfloat16* dst = nullptr;
    dev_alloc((void**)&dst, (size_t)numel * 2);
    m->owned.push_back(dst);
    kernels::f32_to_bf16(src, dst, numel, m->stream);
    MB_CUDA(cudaStreamSynchronize(m->stream));
    cudaFree(m->raw[name].p);
    m->raw.erase(name);
    return dst;
}

void build_clip_layers(b200_model* m, TowerW& T, const std::string& prefix) {
    const long long w = T.d.width, mlp = T.d.mlp;
    T.layers.resize(T.d.layers);
    for (int i = 0; i < T.d.layers; ++i) {
        const std::string p = prefix + "transformer.resblocks." + std::to_string(i) + ".";
        LayerW& L = T.layers[i];
        L.ln1_w = param(m, p + "ln_1.weight", w);
        L.ln1_b = param(m, p + "ln_1.bias", w);
        L.w_qkv = to_bf16(m, p + "attn.in_proj_weight", 3 * w * w);
        L.b_qkv = param(m, p + "attn.in_proj_bias", 3 * w);
        L.w_o = to_bf16(m, p + "attn.out_proj.weight", w * w);
        L.b_o = param(m, p + "attn.out_proj.bias", w);
        L.ln2_w = param(m, p + "ln_2.weight", w);
        L.ln2_b = param(m, p + "ln_2.bias", w);
        L.w_fc = to_bf16(m, p + "mlp.c_fc.weight", mlp * w);
        L.b_fc = param(m, p + "mlp.c_fc.bias", mlp);
        L.w_proj = to_bf16(m, p + "mlp.c_proj.weight", w * mlp);
        L.b_proj = param(m, p + "mlp.c_proj.bias", w);
    }
}

// HF parameter names of a post-LN layer below "encoder.layer.N.": BertLayer and MPNetLayer differ in the attention part
struct PostLnNames {
    const char* qkv[3];   // query / key / value Linear
    const char* out;      // attention output Linear
    const char* ln1;      // LayerNorm after attention
};
constexpr PostLnNames BERT_NAMES{{"attention.self.query", "attention.self.key", "attention.self.value"},
                                 "attention.output.dense", "attention.output.LayerNorm"};
constexpr PostLnNames MPNET_NAMES{{"attention.attn.q", "attention.attn.k", "attention.attn.v"}, "attention.attn.o",
                                  "attention.LayerNorm"};

void build_bert_layers(b200_model* m, TowerW& T, const PostLnNames& nm = BERT_NAMES) {
    const long long w = T.d.width, mlp = T.d.mlp;
    T.layers.resize(T.d.layers);
    for (int i = 0; i < T.d.layers; ++i) {
        const std::string p = "encoder.layer." + std::to_string(i) + ".";
        LayerW& L = T.layers[i];
        // fuse query / key / value into one [3w, w] weight and one [3w] bias
        __nv_bfloat16* wq = nullptr;
        float* bq = nullptr;
        dev_alloc((void**)&wq, (size_t)3 * w * w * 2);
        dev_alloc((void**)&bq, (size_t)3 * w * 4);
        m->owned.push_back(wq);
        m->owned.push_back(bq);
        for (int j = 0; j < 3; ++j) {
            const std::string base = p + nm.qkv[j];
            kernels::f32_to_bf16(param(m, base + ".weight", w * w), wq + (size_t)j * w * w, w * w, m->stream);
            MB_CUDA(cudaMemcpyAsync(bq + (size_t)j * w, param(m, base + ".bias", w), (size_t)w * 4, cudaMemcpyDeviceToDevice,
                                    m->stream));
        }
        MB_CUDA(cudaStreamSynchronize(m->stream));
        for (int j = 0; j < 3; ++j) {
            const std::string wn = p + nm.qkv[j] + ".weight";
            cudaFree(m->raw[wn].p);
            m->raw.erase(wn);
        }
        L.w_qkv = wq;
        L.b_qkv = bq;
        L.w_o = to_bf16(m, p + nm.out + ".weight", w * w);
        L.b_o = param(m, p + nm.out + ".bias", w);
        L.ln1_w = param(m, p + nm.ln1 + ".weight", w);  // post-LN after attention
        L.ln1_b = param(m, p + nm.ln1 + ".bias", w);
        L.w_fc = to_bf16(m, p + "intermediate.dense.weight", mlp * w);
        L.b_fc = param(m, p + "intermediate.dense.bias", mlp);
        L.w_proj = to_bf16(m, p + "output.dense.weight", w * mlp);
        L.b_proj = param(m, p + "output.dense.bias", w);
        L.ln2_w = param(m, p + "output.LayerNorm.weight", w);  // post-LN after the MLP
        L.ln2_b = param(m, p + "output.LayerNorm.bias", w);
    }
}

struct Counter {
    int n = 0;
};

struct ProfScope {
    b200_model* m;
    bool on;
    ProfScope(b200_model* mm, int cls) : m(mm), on(mm->profiling) {
        if (!on) return;
        if ((size_t)(2 * m->prof_n + 2) > m->prof_ev.size()) {
            for (int i = 0; i < 64; ++i) {
                cudaEvent_t e;
                MB_CUDA(cudaEventCreate(&e));
                m->prof_ev.push_back(e);
            }
            m->prof_cls.resize(m->prof_ev.size() / 2);
        }
        m->prof_cls[m->prof_n] = cls;
        MB_CUDA(cudaEventRecord(m->prof_ev[2 * m->prof_n], m->stream));
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(m->prof_ev[2 * m->prof_n + 1], m->stream);
        ++m->prof_n;
    }
};

void linear(b200_model* m, Counter& c, const __nv_bfloat16* A, int M, int K, const __nv_bfloat16* W, int N,
            const gemm::Epilogue& ep) {
    ProfScope ps(m, 0);
    gemm::launch(A, K, W, M, N, K, ep, m->sms, m->stream);
    ++c.n;
}

void attend(b200_model* m, Counter& c, int B, int S, int w, int heads, int mask_mode, const int32_t* kv_len,
            const float* bias_log2 = nullptr) {
    ProfScope ps(m, 1);
    c.n += attention::launch(m->qkv, m->o, B, S, w, heads, mask_mode, kv_len, bias_log2, m->stream);
}

// Pre-LN residual blocks (open_clip ResidualAttentionBlock).  x (fp32) is the residual stream, h (bf16) the LayerNorm
// output the next GEMM consumes.
void run_clip_blocks(b200_model* m, Counter& c, const TowerW& T, int B, int S, int mask_mode) {
    const int M = B * S, w = T.d.width, mlp = T.d.mlp;
    const int act = m->desc.act == B200_ACT_QUICKGELU ? gemm::ACT_QUICKGELU : gemm::ACT_GELU;
    for (const LayerW& L : T.layers) {
        kernels::layernorm(m->x, w, L.ln1_w, L.ln1_b, 1e-5f, M, w, nullptr, m->h, m->stream);
        ++c.n;
        gemm::Epilogue e1;
        e1.bias = L.b_qkv;
        e1.out = m->qkv;
        e1.ldo = 3 * w;
        linear(m, c, m->h, M, w, L.w_qkv, 3 * w, e1);
        attend(m, c, B, S, w, T.d.heads, mask_mode, nullptr);
        gemm::Epilogue e2;
        e2.bias = L.b_o;
        e2.residual = m->x;
        e2.ldr = w;
        e2.out = m->x;
        e2.ldo = w;
        e2.out_fp32 = 1;
        linear(m, c, m->o, M, w, L.w_o, w, e2);
        kernels::layernorm(m->x, w, L.ln2_w, L.ln2_b, 1e-5f, M, w, nullptr, m->h, m->stream);
        ++c.n;
        gemm::Epilogue e3;
        e3.bias = L.b_fc;
        e3.act = act;
        e3.out = m->u;
        e3.ldo = mlp;
        linear(m, c, m->h, M, w, L.w_fc, mlp, e3);
        gemm::Epilogue e4;
        e4.bias = L.b_proj;
        e4.residual = m->x;
        e4.ldr = w;
        e4.out = m->x;
        e4.ldo = w;
        e4.out_fp32 = 1;
        linear(m, c, m->u, M, mlp, L.w_proj, w, e4);
    }
}

// Post-LN blocks (HF BertLayer / MPNetLayer); on entry x (fp32) and h (bf16) both hold the embedding LayerNorm output.
// Both LayerNorms of a layer follow the GEMM before them and rewrite x in place.  eps: 1e-12 for BERT, 1e-5 for MPNet;
// T.rel_bias (MPNet) is added to every attention score.
void run_bert_blocks(b200_model* m, Counter& c, const TowerW& T, int B, int S, float eps) {
    const int M = B * S, w = T.d.width, mlp = T.d.mlp;
    for (const LayerW& L : T.layers) {
        gemm::Epilogue e1;
        e1.bias = L.b_qkv;
        e1.out = m->qkv;
        e1.ldo = 3 * w;
        linear(m, c, m->h, M, w, L.w_qkv, 3 * w, e1);
        attend(m, c, B, S, w, T.d.heads, attention::MASK_KEYLEN, m->aux, T.rel_bias);
        gemm::Epilogue e2;
        e2.bias = L.b_o;
        e2.residual = m->x;
        e2.ldr = w;
        e2.out = m->x;
        e2.ldo = w;
        e2.out_fp32 = 1;
        linear(m, c, m->o, M, w, L.w_o, w, e2);
        kernels::layernorm(m->x, w, L.ln1_w, L.ln1_b, eps, M, w, m->x, m->h, m->stream);
        ++c.n;
        gemm::Epilogue e3;
        e3.bias = L.b_fc;
        e3.act = gemm::ACT_GELU;
        e3.out = m->u;
        e3.ldo = mlp;
        linear(m, c, m->h, M, w, L.w_fc, mlp, e3);
        gemm::Epilogue e4;
        e4.bias = L.b_proj;
        e4.residual = m->x;
        e4.ldr = w;
        e4.out = m->x;
        e4.ldo = w;
        e4.out_fp32 = 1;
        linear(m, c, m->u, M, mlp, L.w_proj, w, e4);
        kernels::layernorm(m->x, w, L.ln2_w, L.ln2_b, eps, M, w, m->x, m->h, m->stream);
        ++c.n;
    }
}

// images already as device uint8 [n, S, S, 3] (u8 != nullptr) or device fp32 CHW (f32 != nullptr)
// MPNet's LayerNorm eps (layer_norm_eps of the all-mpnet-base-v2 family's config.json; transformers' MPNetConfig
// default is 1e-12)
constexpr float MPNET_LN_EPS = 1e-5f;

void forward_images_eager(b200_model* m, Counter& c, const uint8_t* u8, const float* f32, int n, int normalize,
                          float* d_out) {
    const TowerW& T = m->vision;
    const int S = T.d.image_size, p = T.d.patch, w = T.d.width, G = T.grid * T.grid;
    gemm::Epilogue e;  // conv1 (no bias) + positional embedding, scattered to token rows 1..G of each image
    e.out = m->x;
    e.ldo = w;
    e.out_fp32 = 1;
    e.remap_group = G;
    e.rowbias = T.pos;
    if (u8 && T.conv_wg && (reinterpret_cast<uintptr_t>(u8) & 15) == 0) {
        // uint8 pixels -> ToTensor + Normalize -> bf16 inside the GEMM's operand load: no patch matrix in HBM
        gemm::PatchGather pg;
        pg.img = u8;
        pg.n = n;
        pg.S = S;
        pg.patch = p;
        for (int i = 0; i < 3; ++i) {
            pg.mean[i] = m->desc.image_mean[i];
            pg.std[i] = m->desc.image_std[i];
        }
        ProfScope ps(m, 0);
        gemm::launch_patch_embed(pg, T.conv_wg, w, e, m->sms, m->stream);
        ++c.n;
    } else {
        // preprocessed fp32 CHW tensors (the reference's parity path) and shapes the gather does not cover
        if (!m->patches) dev_alloc((void**)&m->patches, (size_t)m->desc.max_batch * G * T.kpad * 2);
        if (u8)
            kernels::im2col_u8(u8, n, S, p, T.kpad, m->desc.image_mean, m->desc.image_std, m->patches, m->stream);
        else
            kernels::im2col_f32(f32, n, S, p, T.kpad, m->patches, m->stream);
        linear(m, c, m->patches, n * G, T.kpad, T.conv_w, w, e);
        ++c.n;
    }
    kernels::vit_cls_rows(m->x, T.cls, T.pos, n, T.tokens, w, m->stream);
    kernels::layernorm(m->x, w, T.ln_pre_w, T.ln_pre_b, 1e-5f, n * T.tokens, w, m->x, nullptr, m->stream);
    c.n += 2;
    run_clip_blocks(m, c, T, n, T.tokens, attention::MASK_NONE);
    kernels::clip_head(m->x, T.tokens, nullptr, T.ln_out_w, T.ln_out_b, 1e-5f, T.proj, n, w, m->desc.embed_dim, normalize,
                       d_out, m->pooled, m->stream);
    c.n += 3;
}

void forward_tokens_eager(b200_model* m, Counter& c, const int32_t* d_ids, const int32_t* d_mask, int n, int S,
                          int normalize, float* d_out) {
    const TowerW& T = m->text;
    const int w = T.d.width;
    if (m->desc.arch == B200_ARCH_CLIP) {
        kernels::clip_text_embed(d_ids, T.tok, T.pos, n, S, w, T.d.vocab, m->x, m->aux, m->stream);
        c.n += 1;
        run_clip_blocks(m, c, T, n, S, attention::MASK_CAUSAL);
        kernels::clip_head(m->x, S, m->aux, T.ln_out_w, T.ln_out_b, 1e-5f, T.proj, n, w, m->desc.embed_dim, normalize,
                           d_out, m->pooled, m->stream);
        c.n += 3;
    } else if (m->desc.arch == B200_ARCH_MPNET) {
        kernels::mpnet_embed_ln(d_ids, d_mask, T.tok, T.pos, T.emb_ln_w, T.emb_ln_b, MPNET_LN_EPS, n, S, w, T.d.vocab,
                                m->x, m->h, m->aux, m->stream);
        c.n += 1;
        run_bert_blocks(m, c, T, n, S, MPNET_LN_EPS);
        kernels::bert_head(m->x, m->aux, n, S, w, m->desc.pool, normalize, d_out, m->stream);
        c.n += 1;
    } else {
        kernels::bert_embed_ln(d_ids, d_mask, T.tok, T.pos, T.type0, T.emb_ln_w, T.emb_ln_b, 1e-12f, n, S, w, T.d.vocab,
                               m->x, m->h, m->aux, m->stream);
        c.n += 1;
        run_bert_blocks(m, c, T, n, S, 1e-12f);
        kernels::bert_head(m->x, m->aux, n, S, w, m->desc.pool, normalize, d_out, m->stream);
        c.n += 1;
    }
}

// Small batches (a single query, a handful of chunks) are launch-bound: ~90-180 kernels of a few microseconds each,
// every GEMM launch also encoding two tensor maps on the host.  The first call of a shape runs eagerly (one-time
// attribute set-up happens there), the second is captured into a CUDA graph, later ones replay it.
constexpr long long GRAPH_MAX_TOKENS = 8192;
constexpr size_t GRAPH_MAX_ENTRIES = 64;

template <class Body>
void run_graphed(b200_model* m, Counter& c, const b200_model::GraphKey& key, long long tokens, Body&& body) {
    static const bool disabled = getenv("MARQO_B200_NO_GRAPHS") != nullptr;   // kill switch / A-B timing
    if (disabled || tokens > GRAPH_MAX_TOKENS || m->profiling || m->external_stream) {
        body(c);
        return;
    }
    auto it = m->graphs.find(key);
    if (it == m->graphs.end()) {
        if (m->graphs.size() < GRAPH_MAX_ENTRIES) m->graphs[key] = b200_model::GraphEntry{};
        body(c);
        return;
    }
    if (!it->second.exec) {
        Counter cc;
        MB_CUDA(cudaStreamBeginCapture(m->stream, cudaStreamCaptureModeThreadLocal));
        cudaGraph_t graph = nullptr;
        try {
            body(cc);
        } catch (...) {
            cudaStreamEndCapture(m->stream, &graph);
            if (graph) cudaGraphDestroy(graph);
            m->graphs.erase(it);
            throw;
        }
        MB_CUDA(cudaStreamEndCapture(m->stream, &graph));
        cudaGraphExec_t exec = nullptr;
        const cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        MB_CUDA(e);
        it->second.exec = exec;
        it->second.launches = cc.n;
    }
    MB_CUDA(cudaGraphLaunch(it->second.exec, m->stream));
    c.n += it->second.launches;
}

void ensure_in_dev(b200_model* m, size_t bytes) {
    if (bytes <= m->in_dev_bytes) return;
    cudaFree(m->in_dev);
    m->in_dev = nullptr;
    m->in_dev_bytes = 0;
    dev_alloc(&m->in_dev, bytes);
    m->in_dev_bytes = bytes;
}

void forward_images(b200_model* m, Counter& c, const uint8_t* u8, const float* f32, int n, int normalize, float* d_out) {
    const b200_model::GraphKey key{0, n, 0, normalize, u8, f32, d_out};
    run_graphed(m, c, key, (long long)n * m->vision.tokens,
                [&](Counter& cc) { forward_images_eager(m, cc, u8, f32, n, normalize, d_out); });
}

void forward_tokens(b200_model* m, Counter& c, const int32_t* d_ids, const int32_t* d_mask, int n, int S, int normalize,
                    float* d_out) {
    const b200_model::GraphKey key{1, n, S, normalize, d_ids, d_mask, d_out};
    run_graphed(m, c, key, (long long)n * S,
                [&](Counter& cc) { forward_tokens_eager(m, cc, d_ids, d_mask, n, S, normalize, d_out); });
}

void require_ready(b200_model* m) {
    MB_CHECK_ARG(m != nullptr, "model is NULL");
    if (!m->finalized) fail(B200_ERR_INVALID_ARG, "b200_model_finalize has not been called");
}

int batch_cap_tokens(b200_model* m, int tokens_per_item) {
    return (int)std::max<long long>(1, std::min<long long>(m->desc.max_batch, m->max_tokens / tokens_per_item));
}

struct TimedRegion {
    b200_model* m;
    Counter c;
    explicit TimedRegion(b200_model* mm) : m(mm) { MB_CUDA(cudaEventRecord(m->ev0, m->stream)); }
    void finish() {
        MB_CUDA(cudaEventRecord(m->ev1, m->stream));
        m->timing_valid = true;
        m->last_launches = c.n;
    }
};

// device-resident uint8 images of size h x w -> embeddings
void encode_images_u8_dev(b200_model* m, Counter& c, const uint8_t* d_img, int n, int h, int w, int normalize,
                          float* d_out) {
    const TowerW& T = m->vision;
    const int S = T.d.image_size;
    const int cap = batch_cap_tokens(m, T.tokens);
    for (int o = 0; o < n; o += cap) {
        const int nb = std::min(cap, n - o);
        const uint8_t* src = d_img + (size_t)o * h * w * 3;
        if (h != S || w != S) {
            kernels::resize_crop_u8(src, nb, h, w, S, m->resized, m->stream);
            c.n += 2;
            src = m->resized;
        }
        forward_images(m, c, src, nullptr, nb, normalize, d_out + (size_t)o * m->desc.embed_dim);
    }
}

void encode_tokens_dev(b200_model* m, Counter& c, const int32_t* d_ids, const int32_t* d_mask, int n, int S, int normalize,
                       float* d_out) {
    const int cap = batch_cap_tokens(m, S);
    for (int o = 0; o < n; o += cap) {
        const int nb = std::min(cap, n - o);
        forward_tokens(m, c, d_ids + (size_t)o * S, d_mask ? d_mask + (size_t)o * S : nullptr, nb, S, normalize,
                       d_out + (size_t)o * m->desc.embed_dim);
    }
}

void check_tokens_args(b200_model* m, int n, int S) {
    MB_CHECK_ARG(m->text.present, "this model has no text tower");
    MB_CHECK_ARG(n > 0, "n must be positive");
    MB_CHECK_ARG(S > 0 && S <= m->text.max_pos, "sequence length %d out of range (1..%d)", S, m->text.max_pos);
}

}  // namespace

extern "C" {

int b200_model_create(int device, const b200_model_desc* desc, b200_model** out) {
    return guarded([&] {
        MB_CHECK_ARG(desc && out, "NULL argument");
        *out = nullptr;
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
            cudaGetLastError();
            fail(B200_ERR_NO_DEVICE, "no CUDA device available (marqo_b200 has no CPU fallback)");
        }
        MB_CHECK_ARG(device >= 0 && device < ndev, "device %d out of range (%d devices)", device, ndev);
        int major = 0;
        MB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
        if (major != 10) fail(B200_ERR_NO_DEVICE, "device %d has compute capability %d.x; sm_100 required", device, major);
        MB_CHECK_ARG(desc->arch == B200_ARCH_CLIP || desc->arch == B200_ARCH_BERT || desc->arch == B200_ARCH_MPNET,
                     "unknown arch %d", desc->arch);
        MB_CHECK_ARG(desc->max_batch > 0, "max_batch must be positive");
        MB_CHECK_ARG(desc->embed_dim > 0 && desc->embed_dim <= 4096, "embed_dim out of range");
        const bool has_vision = desc->arch == B200_ARCH_CLIP && desc->vision.layers > 0;
        const bool has_text = desc->text.layers > 0;
        MB_CHECK_ARG(has_vision || has_text, "model has no tower");
        if (has_vision) {
            check_tower(desc->vision, "vision");
            MB_CHECK_ARG(desc->vision.patch > 0 && desc->vision.image_size % desc->vision.patch == 0,
                         "image_size must be a multiple of patch");
            for (int i = 0; i < 3; ++i) MB_CHECK_ARG(desc->image_std[i] > 0.f, "image_std must be positive");
        }
        if (has_text) {
            check_tower(desc->text, "text");
            MB_CHECK_ARG(desc->text.ctx > 0 && desc->text.vocab > 0, "text.ctx and text.vocab must be positive");
            if (desc->arch == B200_ARCH_BERT)
                MB_CHECK_ARG(desc->embed_dim == desc->text.width, "BERT embed_dim must equal width");
            if (desc->arch == B200_ARCH_MPNET) {
                MB_CHECK_ARG(desc->embed_dim == desc->text.width, "MPNet embed_dim must equal width");
                MB_CHECK_ARG(desc->text.ctx > 2, "MPNet text.ctx (max_position_embeddings) must exceed 2");
            }
        }
        DeviceGuard g(device);
        b200_model* m = new b200_model();
        try {
            m->device = device;
            m->desc = *desc;
            m->sms = sm_count(device);
            MB_CUDA(cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking));
            m->stream = m->own_stream;
            MB_CUDA(cudaEventCreate(&m->ev0));
            MB_CUDA(cudaEventCreate(&m->ev1));
            m->vision.present = has_vision;
            m->vision.d = desc->vision;
            m->text.present = has_text;
            m->text.d = desc->text;
            gemm::configure();
        } catch (...) {
            model_free(m);
            throw;
        }
        *out = m;
    });
}

int b200_model_destroy(b200_model* m) {
    return guarded([&] { model_free(m); });
}

int b200_model_load_tensor(b200_model* m, const char* name, const float* data, int64_t numel) {
    return guarded([&] {
        MB_CHECK_ARG(m && name && data, "NULL argument");
        MB_CHECK_ARG(numel > 0, "numel must be positive");
        std::lock_guard<std::mutex> lk(m->mu);
        if (m->finalized) fail(B200_ERR_INVALID_ARG, "model is already finalized");
        DeviceGuard g(m->device);
        Buf b;
        b.bytes = (size_t)numel * sizeof(float);
        dev_alloc(&b.p, b.bytes);
        cudaError_t e = cudaMemcpy(b.p, data, b.bytes, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            cudaFree(b.p);
            MB_CUDA(e);
        }
        auto it = m->raw.find(name);
        if (it != m->raw.end()) {
            cudaFree(it->second.p);
            m->raw.erase(it);
        }
        m->raw[name] = b;
    });
}

int b200_model_finalize(b200_model* m) {
    return guarded([&] {
        MB_CHECK_ARG(m != nullptr, "model is NULL");
        std::lock_guard<std::mutex> lk(m->mu);
        if (m->finalized) return;
        DeviceGuard g(m->device);
        const int E = m->desc.embed_dim;
        long long max_tok = 0, max_w = 0, max_mlp = 0;
        if (m->vision.present) {
            TowerW& T = m->vision;
            const long long w = T.d.width, p = T.d.patch;
            T.grid = T.d.image_size / T.d.patch;
            T.tokens = T.grid * T.grid + 1;
            const int K = 3 * (int)p * (int)p;
            T.kpad = (int)round_up((size_t)K, 64);
            const float* conv = param(m, "visual.conv1.weight", w * K);
            __nv_bfloat16* cw = nullptr;
            dev_alloc((void**)&cw, (size_t)w * T.kpad * 2);
            m->owned.push_back(cw);
            kernels::pad_rows_to_bf16(conv, (int)w, K, T.kpad, cw, m->stream);
            MB_CUDA(cudaStreamSynchronize(m->stream));
            T.conv_w = cw;
            if (gemm::patch_gather_supported(T.d.image_size, (int)p)) {
                __nv_bfloat16* cg = nullptr;
                dev_alloc((void**)&cg, (size_t)w * gemm::patch_gather_k((int)p) * 2);
                m->owned.push_back(cg);
                kernels::patch_weight_rows(conv, (int)w, (int)p, gemm::patch_gather_kbpd((int)p), cg, m->stream);
                MB_CUDA(cudaStreamSynchronize(m->stream));
                T.conv_wg = cg;
            }
            T.cls = param(m, "visual.class_embedding", w);
            T.pos = param(m, "visual.positional_embedding", (long long)T.tokens * w);
            T.ln_pre_w = param(m, "visual.ln_pre.weight", w);
            T.ln_pre_b = param(m, "visual.ln_pre.bias", w);
            build_clip_layers(m, T, "visual.");
            T.ln_out_w = param(m, "visual.ln_post.weight", w);
            T.ln_out_b = param(m, "visual.ln_post.bias", w);
            T.proj = param(m, "visual.proj", w * E);
            max_tok = std::max(max_tok, (long long)m->desc.max_batch * T.tokens);
            max_w = std::max(max_w, w);
            max_mlp = std::max(max_mlp, (long long)T.d.mlp);
            // the bf16 patch matrix of the im2col path is allocated on first use (fp32 CHW input / unsupported shapes)
            if (!T.conv_wg)
                dev_alloc((void**)&m->patches, (size_t)m->desc.max_batch * T.grid * T.grid * T.kpad * 2);
            dev_alloc((void**)&m->resized, (size_t)m->desc.max_batch * T.d.image_size * T.d.image_size * 3);
        }
        if (m->text.present) {
            TowerW& T = m->text;
            const long long w = T.d.width;
            T.max_pos = T.d.ctx;
            if (m->desc.arch == B200_ARCH_CLIP) {
                T.tok = param(m, "token_embedding.weight", (long long)T.d.vocab * w);
                T.pos = param(m, "positional_embedding", (long long)T.d.ctx * w);
                build_clip_layers(m, T, "");
                T.ln_out_w = param(m, "ln_final.weight", w);
                T.ln_out_b = param(m, "ln_final.bias", w);
                T.proj = param(m, "text_projection", w * E);
            } else if (m->desc.arch == B200_ARCH_MPNET) {
                T.max_pos = T.d.ctx - 2;   // position ids 2 .. S + 1
                T.tok = param(m, "embeddings.word_embeddings.weight", (long long)T.d.vocab * w);
                T.pos = param(m, "embeddings.position_embeddings.weight", (long long)T.d.ctx * w);
                T.emb_ln_w = param(m, "embeddings.LayerNorm.weight", w);
                T.emb_ln_b = param(m, "embeddings.LayerNorm.bias", w);
                build_bert_layers(m, T, MPNET_NAMES);
                // [32 buckets, heads] -> the attention kernels' per-head rows over d = key - query (host fold)
                const int H = T.d.heads;
                const float* rb = param(m, "encoder.relative_attention_bias.weight", (long long)attention::REL_BUCKETS * H);
                std::vector<float> rel((size_t)attention::REL_BUCKETS * H), folded((size_t)H * attention::REL_T);
                MB_CUDA(cudaMemcpy(rel.data(), rb, rel.size() * 4, cudaMemcpyDeviceToHost));
                attention::fold_relative_bias(rel.data(), H, T.max_pos - 1, folded.data());
                float* tbl = nullptr;
                dev_alloc((void**)&tbl, folded.size() * 4);
                m->owned.push_back(tbl);
                MB_CUDA(cudaMemcpy(tbl, folded.data(), folded.size() * 4, cudaMemcpyHostToDevice));
                T.rel_bias = tbl;
            } else {
                T.tok = param(m, "embeddings.word_embeddings.weight", (long long)T.d.vocab * w);
                T.pos = param(m, "embeddings.position_embeddings.weight", (long long)T.d.ctx * w);
                const int tv = std::max(1, m->desc.type_vocab);
                T.type0 = param(m, "embeddings.token_type_embeddings.weight", (long long)tv * w);  // row 0 is used
                T.emb_ln_w = param(m, "embeddings.LayerNorm.weight", w);
                T.emb_ln_b = param(m, "embeddings.LayerNorm.bias", w);
                build_bert_layers(m, T);
            }
            max_tok = std::max(max_tok, (long long)m->desc.max_batch * T.d.ctx);
            max_w = std::max(max_w, w);
            max_mlp = std::max(max_mlp, (long long)T.d.mlp);
        }
        // cap the workspace at ~24 GB of activations: larger calls are processed in sub-batches
        const long long bytes_per_tok = max_w * (4 + 2 + 6 + 2) + max_mlp * 2;
        const long long cap_tok = (24LL << 30) / bytes_per_tok;
        m->max_tokens = std::min(max_tok, std::max<long long>(cap_tok, 1024));
        dev_alloc((void**)&m->x, (size_t)m->max_tokens * max_w * 4);
        dev_alloc((void**)&m->h, (size_t)m->max_tokens * max_w * 2);
        dev_alloc((void**)&m->qkv, (size_t)m->max_tokens * max_w * 6);
        dev_alloc((void**)&m->o, (size_t)m->max_tokens * max_w * 2);
        dev_alloc((void**)&m->u, (size_t)m->max_tokens * max_mlp * 2);
        dev_alloc((void**)&m->aux, (size_t)m->desc.max_batch * 4);
        dev_alloc((void**)&m->out_dev, (size_t)m->desc.max_batch * E * 4);
        dev_alloc((void**)&m->pooled, (size_t)m->desc.max_batch * max_w * 4);
        MB_CUDA(cudaStreamSynchronize(m->stream));
        m->finalized = true;
    });
}

int b200_model_encode_images_u8(b200_model* m, const uint8_t* hwc, int n, int h, int w, int normalize, float* out) {
    return guarded([&] {
        require_ready(m);
        MB_CHECK_ARG(hwc && out, "NULL buffer");
        MB_CHECK_ARG(m->vision.present, "this model has no vision tower");
        MB_CHECK_ARG(n > 0 && h > 0 && w > 0, "n, h, w must be positive");
        std::lock_guard<std::mutex> lk(m->mu);
        DeviceGuard g(m->device);
        const int E = m->desc.embed_dim;
        const int cap = m->desc.max_batch;
        const size_t img_bytes = (size_t)h * w * 3;
        ensure_in_dev(m, (size_t)std::min(n, cap) * img_bytes);
        TimedRegion tr(m);
        for (int o = 0; o < n; o += cap) {
            const int nb = std::min(cap, n - o);
            MB_CUDA(cudaMemcpyAsync(m->in_dev, hwc + (size_t)o * img_bytes, (size_t)nb * img_bytes, cudaMemcpyHostToDevice,
                                    m->stream));
            encode_images_u8_dev(m, tr.c, reinterpret_cast<const uint8_t*>(m->in_dev), nb, h, w, normalize, m->out_dev);
            MB_CUDA(cudaMemcpyAsync(out + (size_t)o * E, m->out_dev, (size_t)nb * E * 4, cudaMemcpyDeviceToHost, m->stream));
            MB_CUDA(cudaStreamSynchronize(m->stream));
        }
        tr.finish();
    });
}

int b200_model_encode_images_f32(b200_model* m, const float* chw, int n, int normalize, float* out) {
    return guarded([&] {
        require_ready(m);
        MB_CHECK_ARG(chw && out, "NULL buffer");
        MB_CHECK_ARG(m->vision.present, "this model has no vision tower");
        MB_CHECK_ARG(n > 0, "n must be positive");
        std::lock_guard<std::mutex> lk(m->mu);
        DeviceGuard g(m->device);
        const int E = m->desc.embed_dim, S = m->vision.d.image_size;
        const int cap = batch_cap_tokens(m, m->vision.tokens);
        const size_t img_bytes = (size_t)3 * S * S * 4;
        ensure_in_dev(m, (size_t)std::min(n, cap) * img_bytes);
        TimedRegion tr(m);
        for (int o = 0; o < n; o += cap) {
            const int nb = std::min(cap, n - o);
            MB_CUDA(cudaMemcpyAsync(m->in_dev, chw + (size_t)o * 3 * S * S, (size_t)nb * img_bytes, cudaMemcpyHostToDevice,
                                    m->stream));
            forward_images(m, tr.c, nullptr, reinterpret_cast<const float*>(m->in_dev), nb, normalize, m->out_dev);
            MB_CUDA(cudaMemcpyAsync(out + (size_t)o * E, m->out_dev, (size_t)nb * E * 4, cudaMemcpyDeviceToHost, m->stream));
            MB_CUDA(cudaStreamSynchronize(m->stream));
        }
        tr.finish();
    });
}

int b200_model_encode_tokens(b200_model* m, const int32_t* ids, const int32_t* attn_mask, int n, int seq, int normalize,
                             float* out) {
    return guarded([&] {
        require_ready(m);
        MB_CHECK_ARG(ids && out, "NULL buffer");
        check_tokens_args(m, n, seq);
        if (attn_mask && (m->desc.arch == B200_ARCH_BERT || m->desc.arch == B200_ARCH_MPNET)) {
            // the kernels implement prefix (right-padded) masks, which is what the tokenizer call at
            // hugging_face_model.py:179-185 produces
            for (int b = 0; b < n; ++b) {
                bool seen_zero = false;
                for (int s = 0; s < seq; ++s) {
                    const bool on = attn_mask[(size_t)b * seq + s] != 0;
                    if (on && seen_zero) fail(B200_ERR_UNSUPPORTED, "attention mask of item %d is not a prefix mask", b);
                    seen_zero |= !on;
                }
            }
        }
        std::lock_guard<std::mutex> lk(m->mu);
        DeviceGuard g(m->device);
        const int E = m->desc.embed_dim;
        const int cap = batch_cap_tokens(m, seq);
        const size_t row_bytes = (size_t)seq * 4;
        ensure_in_dev(m, (size_t)std::min(n, cap) * row_bytes * 2);
        int32_t* d_ids = reinterpret_cast<int32_t*>(m->in_dev);
        int32_t* d_mask = d_ids + (size_t)std::min(n, cap) * seq;
        TimedRegion tr(m);
        for (int o = 0; o < n; o += cap) {
            const int nb = std::min(cap, n - o);
            MB_CUDA(cudaMemcpyAsync(d_ids, ids + (size_t)o * seq, (size_t)nb * row_bytes, cudaMemcpyHostToDevice, m->stream));
            if (attn_mask)
                MB_CUDA(cudaMemcpyAsync(d_mask, attn_mask + (size_t)o * seq, (size_t)nb * row_bytes, cudaMemcpyHostToDevice,
                                        m->stream));
            forward_tokens(m, tr.c, d_ids, attn_mask ? d_mask : nullptr, nb, seq, normalize, m->out_dev);
            MB_CUDA(cudaMemcpyAsync(out + (size_t)o * E, m->out_dev, (size_t)nb * E * 4, cudaMemcpyDeviceToHost, m->stream));
            MB_CUDA(cudaStreamSynchronize(m->stream));
        }
        tr.finish();
    });
}

int b200_model_encode_images_u8_device(b200_model* m, const uint8_t* d_hwc, int n, int h, int w, int normalize,
                                       float* d_out, int sync) {
    return guarded([&] {
        require_ready(m);
        MB_CHECK_ARG(d_hwc && d_out, "NULL buffer");
        MB_CHECK_ARG(m->vision.present, "this model has no vision tower");
        MB_CHECK_ARG(n > 0 && h > 0 && w > 0, "n, h, w must be positive");
        std::lock_guard<std::mutex> lk(m->mu);
        DeviceGuard g(m->device);
        TimedRegion tr(m);
        encode_images_u8_dev(m, tr.c, d_hwc, n, h, w, normalize, d_out);
        tr.finish();
        if (sync) MB_CUDA(cudaStreamSynchronize(m->stream));
    });
}

int b200_model_encode_tokens_device(b200_model* m, const int32_t* d_ids, const int32_t* d_attn_mask, int n, int seq,
                                    int normalize, float* d_out, int sync) {
    return guarded([&] {
        require_ready(m);
        MB_CHECK_ARG(d_ids && d_out, "NULL buffer");
        check_tokens_args(m, n, seq);
        std::lock_guard<std::mutex> lk(m->mu);
        DeviceGuard g(m->device);
        TimedRegion tr(m);
        encode_tokens_dev(m, tr.c, d_ids, d_attn_mask, n, seq, normalize, d_out);
        tr.finish();
        if (sync) MB_CUDA(cudaStreamSynchronize(m->stream));
    });
}

int b200_model_set_stream(b200_model* m, void* cuda_stream, int use_external) {
    return guarded([&] {
        MB_CHECK_ARG(m != nullptr, "model is NULL");
        std::lock_guard<std::mutex> lk(m->mu);
        DeviceGuard g(m->device);
        MB_CUDA(cudaStreamSynchronize(m->stream));
        m->stream = use_external ? reinterpret_cast<cudaStream_t>(cuda_stream) : m->own_stream;
        m->external_stream = use_external != 0;   // a caller's stream may itself be under capture: no graphs there
    });
}

int b200_model_set_profiling(b200_model* m, int enable) {
    return guarded([&] {
        MB_CHECK_ARG(m != nullptr, "model is NULL");
        std::lock_guard<std::mutex> lk(m->mu);
        m->profiling = enable != 0;
        m->prof_n = 0;
    });
}

int b200_model_profile(b200_model* m, float* gemm_ms, int* gemm_launches, float* attention_ms, int* attention_launches) {
    return guarded([&] {
        MB_CHECK_ARG(m && gemm_ms && gemm_launches && attention_ms && attention_launches, "NULL argument");
        std::lock_guard<std::mutex> lk(m->mu);
        DeviceGuard g(m->device);
        float ms[2] = {0.f, 0.f};
        int cnt[2] = {0, 0};
        for (int i = 0; i < m->prof_n; ++i) {
            MB_CUDA(cudaEventSynchronize(m->prof_ev[2 * i + 1]));
            float t = 0.f;
            MB_CUDA(cudaEventElapsedTime(&t, m->prof_ev[2 * i], m->prof_ev[2 * i + 1]));
            ms[m->prof_cls[i]] += t;
            ++cnt[m->prof_cls[i]];
        }
        *gemm_ms = ms[0];
        *gemm_launches = cnt[0];
        *attention_ms = ms[1];
        *attention_launches = cnt[1];
    });
}

int b200_model_last_timing(b200_model* m, float* ms, int* launches) {
    return guarded([&] {
        MB_CHECK_ARG(m && ms && launches, "NULL argument");
        std::lock_guard<std::mutex> lk(m->mu);
        DeviceGuard g(m->device);
        if (!m->timing_valid) fail(B200_ERR_INVALID_ARG, "no encode call has been timed yet");
        MB_CUDA(cudaEventSynchronize(m->ev1));
        MB_CUDA(cudaEventElapsedTime(ms, m->ev0, m->ev1));
        *launches = m->last_launches;
    });
}

}  // extern "C"
