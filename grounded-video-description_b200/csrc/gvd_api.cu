// gvd-b200: C-ABI (include/gvd_b200.h) — model/weight arena, workspace layout, prologue and
// decode orchestration.  Host code only launches kernels; there is no CPU compute path.
#include <atomic>
#include <mutex>
#include <chrono>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/gvd_b200.h"
#include "gvd_kernels.cuh"

// ------------------------------------------------------------------------------------ errors
static thread_local char g_err[1024] = "";
static std::atomic<long long> g_launches{0};
void gvd_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void gvd_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long gvd_launch_count() { return g_launches.load(); }
void gvd_launch_count_add(long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
extern "C" GVD_API const char* gvd_last_error(void) { return g_err; }
extern "C" GVD_API const char* gvd_version(void) { return "gvd-b200 0.1.0 (sm_100a)"; }
extern "C" GVD_API int gvd_op_kernel_launches(void) { return (int)g_launches.load(); }
// backend switches (gvd_set_backend): bit 0 tcgen05 tensor cores for every GEMM-shaped stage (0 = fp32 CUDA cores); bit 1 fused self-attention
// pair; bit 2 (4) 256-column prologue tiles (measured: no gain, off); bit 3 (8) operand-swapped split-K decode products with fused
// reduce + sampler; bit 4 (16) fp16x3 instead of 3xTF32 in the forward GEMMs (pre-split constant weights); bit 5 (32) persistent GRU layer
// kernel (measured: no gain, off); bit 6 (64) programmatic dependent launch in the decode loop (measured: no gain, off); bit 7 (128)
// conversion-free persistent GEMMs for the prologue (activations packed into the fp16x3 image, both operands straight from TMA); bit 8 (256)
// fp16x3 images instead of tf32 planes in the fused self-attention pair; bit 9 (512) pack fusion: the producer of a prologue activation (GEMM
// epilogue / row kernel) stores the fp16x3 operand image the next GEMM streams, instead of a separate pack pass; bit 10 (1024) CTA pairs in
// the persistent prologue GEMM (measured slower: off); bit 11 (2048) thread-per-row epilogue stores in the persistent prologue GEMM (the
// reference its staged epilogue is tested against).
// Default 923 = 1 + 2 + 8 + 16 + 128 + 256 + 512.
static std::atomic<int> g_backend{923};
int gvd_backend() { return g_backend.load(std::memory_order_relaxed); }
// registry of pre-split constant weights (fp16x3 variant): fp32 weight pointer -> packed image
namespace {
struct PackedW { const float* packed; long long ld; int N, K; long long ldw; };
std::mutex g_pw_mu;
std::unordered_map<const float*, PackedW> g_pw;
}  // namespace
bool gvd_packed_lookup(const float* W, long long ldw, int N, int K, const float** packed, long long* ld_packed) {
    std::lock_guard<std::mutex> lk(g_pw_mu);
    auto it = g_pw.find(W);
    if (it == g_pw.end() || it->second.ldw != ldw || it->second.N != N || it->second.K != K) return false;
    *packed = it->second.packed;
    *ld_packed = it->second.ld;
    return true;
}
bool gvd_pdl() { return (g_backend.load(std::memory_order_relaxed) & 64) != 0; }
static thread_local int g_f16_depth = 0;
void gvd_f16_scope(int delta) { g_f16_depth += delta; }
bool gvd_gemm_f16() { return g_f16_depth > 0 && (g_backend.load(std::memory_order_relaxed) & 16) != 0; }
extern "C" GVD_API int gvd_set_backend(int flags) { g_backend.store(flags); return 0; }
extern "C" GVD_API int gvd_get_backend(void) { return g_backend.load(); }

// ------------------------------------------------------------------------------------ stage profiler
// Optional CUDA-event timing of each stage / kernel family ON THE LAUNCHING STREAM (bench.py uses it
// for the per-kernel roofline; off by default: zero events recorded).
#include <mutex>
namespace {
struct ProfRec { const char* name; cudaEvent_t a, b; };
std::atomic<int> g_prof_on{0};
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof_recs;
std::vector<cudaEvent_t> g_prof_pool;
struct ProfAgg { double ms; long long n; };
std::unordered_map<std::string, ProfAgg> g_prof_agg;
cudaEvent_t prof_event() {
    if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
struct ProfScope {
    const char* name; cudaStream_t st; cudaEvent_t a{}, b{}; bool on;
    ProfScope(const char* n, cudaStream_t s) : name(n), st(s), on(g_prof_on.load(std::memory_order_relaxed) != 0) {
        if (!on) return;
        std::lock_guard<std::mutex> lk(g_prof_mu);
        a = prof_event(); b = prof_event();
        cudaEventRecord(a, st);
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(b, st);
        std::lock_guard<std::mutex> lk(g_prof_mu);
        g_prof_recs.push_back({name, a, b});
    }
};
void prof_collect() {      // caller has synchronised the stream(s)
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (auto& r : g_prof_recs) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { auto& g = g_prof_agg[r.name]; g.ms += ms; g.n += 1; }
        g_prof_pool.push_back(r.a); g_prof_pool.push_back(r.b);
    }
    g_prof_recs.clear();
}
}  // namespace
extern "C" GVD_API int gvd_profile_enable(int on) {
    g_prof_on.store(on ? 1 : 0);
    return 0;
}
extern "C" GVD_API int gvd_profile_reset(void) {
    prof_collect();
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_agg.clear();
    return 0;
}
extern "C" GVD_API int gvd_profile_count(void) {
    prof_collect();
    std::lock_guard<std::mutex> lk(g_prof_mu);
    return (int)g_prof_agg.size();
}
extern "C" GVD_API const char* gvd_profile_entry(int i, double* total_ms, long long* count) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    int k = 0;
    for (auto& kv : g_prof_agg) {
        if (k++ == i) { if (total_ms) *total_ms = kv.second.ms; if (count) *count = kv.second.n; return kv.first.c_str(); }
    }
    return nullptr;
}
#define GVD_STAGE(name, expr) do { ProfScope _ps(name, st); GVD_TRY(expr); } while (0)

static inline size_t rup(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int rup4(int x) { return (x + 3) / 4 * 4; }

// ------------------------------------------------------------------------------------ small pack kernels
namespace {
__global__ void relu_copy_kernel(const float* x, float* y, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = fmaxf(x[i], 0.f);
}
__global__ void add2_kernel(const float* a, const float* b, float* y, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = a[i] + b[i];
}
// dst[r, c] = (rmap[r] >= 0 && cmap[c] >= 0) ? src[rmap[r], cmap[c]] : 0 ; identity map when nullptr
__global__ void pack_kernel(float* dst, long long ld_dst, const float* src, long long ld_src, const int* rmap, const int* cmap,
                            int nrows, int ncols) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (c >= ncols || r >= nrows) return;
    const int sr = rmap ? rmap[r] : r, sc = cmap ? cmap[c] : c;
    dst[(long long)r * ld_dst + c] = (sr >= 0 && sc >= 0) ? src[(long long)sr * ld_src + sc] : 0.f;
}
// xt = ReLU(embed[token]) (model.py:79-82,605): materialised once per step for the tensor-core LSTM path
__global__ void embed_relu_kernel(const float* table, const long long* tokens, float* out, long long ld_out, int B, int E, int V, float* pk,
                                  long long ld_pk) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * E) return;                       // B * E is a multiple of 32 whenever pk is given (E % 32 == 0)
    const int b = i / E, e = i % E;
    const long long tok = tokens[b];
    // ids outside the table read as NaN instead of out of bounds (nn.Embedding raises; the Python shim validates host-visible ids)
    const float v = (tok >= 0 && tok < V) ? fmaxf(table[tok * E + e], 0.f) : __int_as_float(0x7fc00000);
    out[(long long)b * ld_out + e] = v;
    if (pk) {                                     // fp16x3 operand image (E even: lanes e, e + 1 sit in one warp)
        const float vn = __shfl_down_sync(0xffffffffu, v, 1);
        if (!(e & 1)) {
            uint32_t hi, lo;
            f16x3_split_pair(v, vn, GVD_F16_SA, hi, lo);
            uint32_t* dst = reinterpret_cast<uint32_t*>(pk) + (long long)b * ld_pk + f16x3_word(e);
            dst[0] = hi; dst[16] = lo;
        }
    }
}
__global__ void bn_affine_kernel(const float* w, const float* b, const float* mean, const float* var, float* scale, float* shift,
                                 int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float s = w[i] / sqrtf(var[i] + 1e-5f);      // BatchNorm1d eval, eps 1e-5 (model.py:114)
    scale[i] = s;
    shift[i] = b[i] - mean[i] * s;
}
}  // namespace

// ------------------------------------------------------------------------------------ model
struct Param { std::string key; size_t numel; size_t off; bool set; };

struct gvd_model {
    gvd_dims_t d;
    int R, G, NC, FCX, FCXp, PIN, PINp, NCp, Vp, HS, HP, nheads, rgb, motion;
    std::vector<int> head_off, head_size;
    std::vector<Param> params;
    std::unordered_map<std::string, int> index;
    float* arena = nullptr;      // raw state_dict entries
    float* packed = nullptr;     // derived operands
    size_t arena_floats = 0, packed_floats = 0;
    bool finalized = false;
    // packed operands
    float *fc_embed_w, *pool_embed_w, *vis_relu, *h2att_w, *h2att_b, *att_bias_sum, *bn_scale, *bn_shift;
    float *w_att_cat, *w_lang_cat;      // [4H, E+H] = [W_ih[:, H:] | W_hh] and [4H, 3H] = [W_ih | W_hh]: one K axis per LSTM (split-K path)
    float *wqk[2], *wv[2], *wo[2];
    float *gru_wih[2], *gru_bih[2], *gru_whh[2], *gru_bhh[2];
    int* maps = nullptr;
    float* packed16 = nullptr;   // fp16x3 images of the constant GEMM weights (gvd_pack_f16x3), registered in g_pw
    std::vector<const float*> pw_keys;
    // host-buffer entry point: second stream + events for the chunked H2D / compute pipeline
    cudaStream_t copy_stream = nullptr;
    std::vector<cudaEvent_t> events;
    // frame branch (P1 + P7) on its own stream, concurrent with the region stages (P2-P6): the bi-GRU is a chain of short
    // launches on 32 SMs that the big GEMMs would otherwise wait behind
    cudaStream_t frame_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // greedy loop captured once per (batch, frames, workspace, backend) as a CUDA graph: 20 steps x 6 launches replayed with one
    // cudaGraphLaunch (no per-launch host cost, back-to-back scheduling on the device)
    cudaStream_t capture_stream = nullptr;
    cudaGraphExec_t greedy_exec = nullptr;
    struct { int B, T, backend; void* ws; size_t ws_bytes; } greedy_key{0, 0, 0, nullptr, 0};
    long long greedy_nodes = 0;      // kernel launches inside one replay (counted while capturing)

    float* P(const std::string& k) const {
        auto it = index.find(k);
        return it == index.end() ? nullptr : arena + params[it->second].off;
    }
};

static void add_param(gvd_model* m, const std::string& key, size_t numel) {
    Param p{key, numel, m->arena_floats, false};
    m->arena_floats += rup(numel, 64);
    m->index[key] = (int)m->params.size();
    m->params.push_back(p);
}

extern "C" GVD_API int gvd_model_create(const gvd_dims_t* dims, gvd_model_t** out) {
    GVD_REQUIRE(dims && out, "model_create: null argument");
    const gvd_dims_t& d = *dims;
    GVD_REQUIRE(d.rnn_size % 4 == 0 && d.rnn_size >= 8 && d.rnn_size <= 1024, "rnn_size must be a multiple of 4 in [8,1024] (got %d)",
                d.rnn_size);
    GVD_REQUIRE(d.rnn_size % 2 == 0 && (d.rnn_size / 2) % 4 == 0, "rnn_size/2 must be a multiple of 4");
    GVD_REQUIRE(d.att_hid_size % 4 == 0 && d.att_hid_size > 0, "att_hid_size must be a multiple of 4");
    GVD_REQUIRE(d.input_encoding_size % 4 == 0 && d.input_encoding_size > 0, "input_encoding_size must be a multiple of 4");
    GVD_REQUIRE(d.att_feat_size == 2048, "att_feat_size must be 2048 (fc7 transfer, misc/model.py:158-178)");
    GVD_REQUIRE(d.fc_feat_size > 2048 && (d.fc_feat_size - 2048) % 4 == 0, "fc_feat_size must be 2048 + motion width");
    GVD_REQUIRE(d.vocab_size >= 2 && d.detect_size >= 1 && d.seq_length >= 1, "bad vocab/detect/seq sizes");
    GVD_REQUIRE(d.num_sampled_frm >= 1 && d.num_prop_per_frm >= 1, "bad proposal grid");
    GVD_REQUIRE(d.unk_idx >= 0 && d.unk_idx < d.vocab_size, "unk_idx out of range");
    gvd_model* m = new gvd_model();
    m->d = d;
    const int H = d.rnn_size, A = d.att_hid_size, E = d.input_encoding_size, V = d.vocab_size, D = d.detect_size;
    m->R = d.num_sampled_frm * d.num_prop_per_frm;
    GVD_REQUIRE(!d.obj_interact || m->R % 4 == 0, "obj_interact needs R %% 4 == 0 (R=%d)", m->R);
    m->G = H / 2;
    m->NC = D + 1;
    m->NCp = rup4(m->NC);
    m->FCX = d.fc_feat_size + 50;
    m->FCXp = rup4(m->FCX);
    m->PIN = d.att_feat_size + 300 + D + 1;
    m->PINp = rup4(m->PIN);
    m->Vp = rup4(V);
    m->rgb = 2048;
    m->motion = d.fc_feat_size - 2048;
    // torch.chunk(6, -1) head split (transformer.py:121): ceil(H/6) each, remainder last
    const int c = (H + 5) / 6;
    for (int o = 0; o < H; o += c) { m->head_off.push_back(o); m->head_size.push_back(std::min(c, H - o)); }
    m->nheads = (int)m->head_off.size();
    m->HS = rup4(c);
    m->HP = m->HS * m->nheads;
    const int G = m->G;
    // the reference state_dict (SURVEY.md 8b), float entries only
    add_param(m, "vis_classifiers_bias", D + 1);
    add_param(m, "loc_fc.0.weight", 300 * 5); add_param(m, "loc_fc.0.bias", 300);
    add_param(m, "embed.0.weight", (size_t)V * E);
    add_param(m, "vis_embed.0.weight", (size_t)(D + 1) * 2048);
    add_param(m, "fc_embed.0.weight", (size_t)H * m->FCX); add_param(m, "fc_embed.0.bias", H);
    add_param(m, "seg_info_embed.0.weight", 50 * 4); add_param(m, "seg_info_embed.0.bias", 50);
    add_param(m, "att_embed.0.0.weight", (size_t)(H / 2) * 2048); add_param(m, "att_embed.0.0.bias", H / 2);
    add_param(m, "att_embed.1.0.weight", (size_t)(H / 2) * m->motion); add_param(m, "att_embed.1.0.bias", H / 2);
    add_param(m, "att_embed_aux.0.weight", H); add_param(m, "att_embed_aux.0.bias", H);
    add_param(m, "att_embed_aux.0.running_mean", H); add_param(m, "att_embed_aux.0.running_var", H);
    add_param(m, "pool_embed.0.weight", (size_t)H * m->PIN); add_param(m, "pool_embed.0.bias", H);
    add_param(m, "ctx2att.weight", (size_t)A * H); add_param(m, "ctx2att.bias", A);
    add_param(m, "ctx2pool.weight", (size_t)A * H); add_param(m, "ctx2pool.bias", A);
    add_param(m, "logit.weight", (size_t)V * H); add_param(m, "logit.bias", V);
    if (d.obj_interact) {
        for (int l = 0; l < 2; ++l) {
            const std::string p = "obj_interact.encoder.layers." + std::to_string(l) + ".";
            for (const char* w : {"wq", "wk", "wv", "wo"}) add_param(m, p + "selfattn.layer." + w + ".weight", (size_t)H * H);
            add_param(m, p + "selfattn.layernorm.gamma", H); add_param(m, p + "selfattn.layernorm.beta", H);
            add_param(m, p + "feedforward.layer.linear1.weight", (size_t)(H / 2) * H); add_param(m, p + "feedforward.layer.linear1.bias", H / 2);
            add_param(m, p + "feedforward.layer.linear2.weight", (size_t)H * (H / 2)); add_param(m, p + "feedforward.layer.linear2.bias", H);
            add_param(m, p + "feedforward.layernorm.gamma", H); add_param(m, p + "feedforward.layernorm.beta", H);
        }
    }
    for (int l = 0; l < 2; ++l)
        for (const char* sfx : {"", "_reverse"}) {
            const std::string s = "_l" + std::to_string(l) + sfx;
            add_param(m, "context_enc.weight_ih" + s, (size_t)3 * G * (l == 0 ? H : 2 * G));
            add_param(m, "context_enc.weight_hh" + s, (size_t)3 * G * G);
            add_param(m, "context_enc.bias_ih" + s, 3 * G);
            add_param(m, "context_enc.bias_hh" + s, 3 * G);
        }
    add_param(m, "ctx2pool_grd.0.weight", (size_t)2048 * d.att_feat_size); add_param(m, "ctx2pool_grd.0.bias", 2048);
    add_param(m, "core.att_lstm.weight_ih", (size_t)4 * H * (E + H)); add_param(m, "core.att_lstm.weight_hh", (size_t)4 * H * H);
    add_param(m, "core.att_lstm.bias_ih", 4 * H); add_param(m, "core.att_lstm.bias_hh", 4 * H);
    add_param(m, "core.lang_lstm.weight_ih", (size_t)4 * H * 2 * H); add_param(m, "core.lang_lstm.weight_hh", (size_t)4 * H * H);
    add_param(m, "core.lang_lstm.bias_ih", 4 * H); add_param(m, "core.lang_lstm.bias_hh", 4 * H);
    for (const char* a : {"attention", "attention2"}) {
        add_param(m, std::string("core.") + a + ".h2att.weight", (size_t)A * H); add_param(m, std::string("core.") + a + ".h2att.bias", A);
        add_param(m, std::string("core.") + a + ".alpha_net.weight", A); add_param(m, std::string("core.") + a + ".alpha_net.bias", 1);
    }
    // present in the checkpoint but never used by the forward pass (AttModel.py:130-131, quirk Q10)
    add_param(m, "core.i2h_2.weight", (size_t)H * 2 * H); add_param(m, "core.i2h_2.bias", H);
    add_param(m, "core.h2h_2.weight", (size_t)H * H); add_param(m, "core.h2h_2.bias", H);

    // packed operand arena
    size_t pf = 0;
    auto take = [&](size_t n) { size_t o = pf; pf += rup(n, 64); return o; };
    std::vector<std::pair<float**, size_t>> slots;
    auto slot = [&](float** p, size_t n) { slots.push_back({p, take(n)}); };
    slot(&m->fc_embed_w, (size_t)H * m->FCXp);
    slot(&m->pool_embed_w, (size_t)H * m->PINp);
    slot(&m->vis_relu, (size_t)m->NC * 2048);
    slot(&m->h2att_w, (size_t)2 * A * H);
    slot(&m->h2att_b, 2 * A);
    slot(&m->att_bias_sum, 4 * H);
    slot(&m->w_att_cat, (size_t)4 * H * (d.input_encoding_size + H));
    slot(&m->w_lang_cat, (size_t)4 * H * 3 * H);
    slot(&m->bn_scale, H);
    slot(&m->bn_shift, H);
    for (int l = 0; l < 2; ++l) {
        if (d.obj_interact) {
            slot(&m->wqk[l], (size_t)3 * m->HP * H);       // [Wq; Wk; Wv] head-padded, one projection GEMM
            slot(&m->wo[l], (size_t)H * m->HP);
        }
        slot(&m->gru_wih[l], (size_t)6 * G * (l == 0 ? H : 2 * G));
        slot(&m->gru_bih[l], 6 * G);
        slot(&m->gru_whh[l], (size_t)6 * G * G);
        slot(&m->gru_bhh[l], 6 * G);
    }
    m->packed_floats = pf;
    if (cudaMalloc(&m->arena, m->arena_floats * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&m->packed, m->packed_floats * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&m->maps, (size_t)(m->HP + 16) * sizeof(int)) != cudaSuccess) {
        gvd_set_error("model_create: cudaMalloc failed (%s)", cudaGetErrorString(cudaGetLastError()));
        gvd_model_destroy(m);
        return 2;
    }
    for (auto& s : slots) *s.first = m->packed + s.second;
    if (d.obj_interact)
        for (int l = 0; l < 2; ++l) m->wv[l] = m->wqk[l] + (size_t)2 * m->HP * H;
    *out = m;
    return 0;
}

extern "C" GVD_API void gvd_model_destroy(gvd_model_t* m) {
    if (!m) return;
    if (m->arena) cudaFree(m->arena);
    if (m->packed) cudaFree(m->packed);
    if (m->maps) cudaFree(m->maps);
    {
        std::lock_guard<std::mutex> lk(g_pw_mu);
        for (const float* k : m->pw_keys) g_pw.erase(k);
    }
    if (m->packed16) cudaFree(m->packed16);
    for (cudaEvent_t e : m->events) cudaEventDestroy(e);
    if (m->copy_stream) cudaStreamDestroy(m->copy_stream);
    if (m->frame_stream) cudaStreamDestroy(m->frame_stream);
    if (m->ev_fork) cudaEventDestroy(m->ev_fork);
    if (m->ev_join) cudaEventDestroy(m->ev_join);
    if (m->greedy_exec) cudaGraphExecDestroy(m->greedy_exec);
    if (m->capture_stream) cudaStreamDestroy(m->capture_stream);
    delete m;
}

extern "C" GVD_API int gvd_model_num_params(const gvd_model_t* m) { return m ? (int)m->params.size() : 0; }
extern "C" GVD_API const char* gvd_model_param_key(const gvd_model_t* m, int i, size_t* numel) {
    if (!m || i < 0 || i >= (int)m->params.size()) return nullptr;
    if (numel) *numel = m->params[i].numel;
    return m->params[i].key.c_str();
}

extern "C" GVD_API int gvd_model_set_param(gvd_model_t* m, const char* key, const float* dev_ptr, size_t numel, void* stream) {
    GVD_REQUIRE(m && key && dev_ptr, "set_param: null argument");
    auto it = m->index.find(key);
    GVD_REQUIRE(it != m->index.end(), "set_param: unexpected key '%s' (not in the reference state_dict for these dims)", key);
    Param& p = m->params[it->second];
    GVD_REQUIRE(p.numel == numel, "set_param: size mismatch for '%s': expected %zu elements, got %zu", key, p.numel, numel);
    GVD_CHECK_CUDA(cudaMemcpyAsync(m->arena + p.off, dev_ptr, numel * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    p.set = true;
    m->finalized = false;
    return 0;
}

static int pack2d(float* dst, long long ld_dst, const float* src, long long ld_src, const int* rmap, const int* cmap, int nrows,
                  int ncols, cudaStream_t st) {
    dim3 grid(gvd_cdiv(ncols, 256), nrows);
    pack_kernel<<<grid, 256, 0, st>>>(dst, ld_dst, src, ld_src, rmap, cmap, nrows, ncols);
    GVD_CHECK_LAUNCH();
    return 0;
}

extern "C" GVD_API int gvd_model_finalize(gvd_model_t* m, void* stream) {
    GVD_REQUIRE(m, "finalize: null model");
    cudaStream_t st = (cudaStream_t)stream;
    for (auto& p : m->params)
        GVD_REQUIRE(p.set || p.key.rfind("core.i2h_2", 0) == 0 || p.key.rfind("core.h2h_2", 0) == 0,
                    "finalize: parameter '%s' was never set (strict load, main.py:638)", p.key.c_str());
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, A = d.att_hid_size, G = m->G;
    // padded-K copies (16-byte row alignment for the 128-bit operand loads)
    GVD_CHECK_CUDA(cudaMemsetAsync(m->fc_embed_w, 0, (size_t)H * m->FCXp * sizeof(float), st));
    GVD_TRY(pack2d(m->fc_embed_w, m->FCXp, m->P("fc_embed.0.weight"), m->FCX, nullptr, nullptr, H, m->FCX, st));
    GVD_CHECK_CUDA(cudaMemsetAsync(m->pool_embed_w, 0, (size_t)H * m->PINp * sizeof(float), st));
    GVD_TRY(pack2d(m->pool_embed_w, m->PINp, m->P("pool_embed.0.weight"), m->PIN, nullptr, nullptr, H, m->PIN, st));
    {   // vis_embed = Embedding + ReLU (model.py:93-97): the class "classifiers" are ReLU(weight)
        const size_t n = (size_t)m->NC * 2048;
        relu_copy_kernel<<<gvd_cdiv(n, 256), 256, 0, st>>>(m->P("vis_embed.0.weight"), m->vis_relu, n);
        GVD_CHECK_LAUNCH();
    }
    GVD_CHECK_CUDA(cudaMemcpyAsync(m->h2att_w, m->P("core.attention.h2att.weight"), (size_t)A * H * 4, cudaMemcpyDeviceToDevice, st));
    GVD_CHECK_CUDA(cudaMemcpyAsync(m->h2att_w + (size_t)A * H, m->P("core.attention2.h2att.weight"), (size_t)A * H * 4, cudaMemcpyDeviceToDevice, st));
    GVD_CHECK_CUDA(cudaMemcpyAsync(m->h2att_b, m->P("core.attention.h2att.bias"), A * 4, cudaMemcpyDeviceToDevice, st));
    GVD_CHECK_CUDA(cudaMemcpyAsync(m->h2att_b + A, m->P("core.attention2.h2att.bias"), A * 4, cudaMemcpyDeviceToDevice, st));
    add2_kernel<<<gvd_cdiv(4 * H, 256), 256, 0, st>>>(m->P("core.att_lstm.bias_ih"), m->P("core.att_lstm.bias_hh"), m->att_bias_sum, 4 * H);
    GVD_CHECK_LAUNCH();
    {   // one K axis per LSTM for the split-K path: [W_ih (token part) | W_hh] and [W_ih | W_hh]
        const int E = d.input_encoding_size;
        GVD_TRY(pack2d(m->w_att_cat, E + H, m->P("core.att_lstm.weight_ih") + H, H + E, nullptr, nullptr, 4 * H, E, st));
        GVD_TRY(pack2d(m->w_att_cat + E, E + H, m->P("core.att_lstm.weight_hh"), H, nullptr, nullptr, 4 * H, H, st));
        GVD_TRY(pack2d(m->w_lang_cat, 3 * H, m->P("core.lang_lstm.weight_ih"), 2 * H, nullptr, nullptr, 4 * H, 2 * H, st));
        GVD_TRY(pack2d(m->w_lang_cat + 2 * H, 3 * H, m->P("core.lang_lstm.weight_hh"), H, nullptr, nullptr, 4 * H, H, st));
    }
    bn_affine_kernel<<<gvd_cdiv(H, 256), 256, 0, st>>>(m->P("att_embed_aux.0.weight"), m->P("att_embed_aux.0.bias"),
                                                        m->P("att_embed_aux.0.running_mean"), m->P("att_embed_aux.0.running_var"),
                                                        m->bn_scale, m->bn_shift, H);
    GVD_CHECK_LAUNCH();
    if (d.obj_interact) {
        // head-padded projections: head h occupies columns [h*HS, h*HS+size_h) (zeros beyond), so every
        // per-head operand starts 16-byte aligned although torch.chunk gives 171/169-wide heads
        std::vector<int> map(m->HP, -1);
        for (int h = 0; h < m->nheads; ++h)
            for (int i = 0; i < m->head_size[h]; ++i) map[h * m->HS + i] = m->head_off[h] + i;
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->maps, map.data(), m->HP * sizeof(int), cudaMemcpyHostToDevice, st));
        GVD_CHECK_CUDA(cudaStreamSynchronize(st));   // `map` is a stack-lifetime host buffer
        for (int l = 0; l < 2; ++l) {
            const std::string p = "obj_interact.encoder.layers." + std::to_string(l) + ".selfattn.layer.";
            GVD_TRY(pack2d(m->wqk[l], H, m->P(p + "wq.weight"), H, m->maps, nullptr, m->HP, H, st));
            GVD_TRY(pack2d(m->wqk[l] + (size_t)m->HP * H, H, m->P(p + "wk.weight"), H, m->maps, nullptr, m->HP, H, st));
            GVD_TRY(pack2d(m->wv[l], H, m->P(p + "wv.weight"), H, m->maps, nullptr, m->HP, H, st));
            GVD_TRY(pack2d(m->wo[l], m->HP, m->P(p + "wo.weight"), H, nullptr, m->maps, H, m->HP, st));
        }
    }
    for (int l = 0; l < 2; ++l) {
        const int in = l == 0 ? H : 2 * G;
        const std::string s = "_l" + std::to_string(l);
        const size_t wsz = (size_t)3 * G * in, hsz = (size_t)3 * G * G;
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->gru_wih[l], m->P("context_enc.weight_ih" + s), wsz * 4, cudaMemcpyDeviceToDevice, st));
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->gru_wih[l] + wsz, m->P("context_enc.weight_ih" + s + "_reverse"), wsz * 4, cudaMemcpyDeviceToDevice, st));
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->gru_bih[l], m->P("context_enc.bias_ih" + s), 3 * G * 4, cudaMemcpyDeviceToDevice, st));
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->gru_bih[l] + 3 * G, m->P("context_enc.bias_ih" + s + "_reverse"), 3 * G * 4, cudaMemcpyDeviceToDevice, st));
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->gru_whh[l], m->P("context_enc.weight_hh" + s), hsz * 4, cudaMemcpyDeviceToDevice, st));
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->gru_whh[l] + hsz, m->P("context_enc.weight_hh" + s + "_reverse"), hsz * 4, cudaMemcpyDeviceToDevice, st));
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->gru_bhh[l], m->P("context_enc.bias_hh" + s), 3 * G * 4, cudaMemcpyDeviceToDevice, st));
        GVD_CHECK_CUDA(cudaMemcpyAsync(m->gru_bhh[l] + 3 * G, m->P("context_enc.bias_hh" + s + "_reverse"), 3 * G * 4, cudaMemcpyDeviceToDevice, st));
    }
    {   // fp16x3 images of every constant weight that is the W operand of a forward GEMM (used when backend bit 4 is set)
        struct Ent { const float* W; long long ldw; int N, K; };
        std::vector<Ent> ents;
        const int E = d.input_encoding_size, V = d.vocab_size;
        ents.push_back({m->P("ctx2pool_grd.0.weight"), d.att_feat_size, 2048, d.att_feat_size});
        ents.push_back({m->vis_relu, 2048, m->NC, 2048});
        ents.push_back({m->pool_embed_w, m->PINp, H, m->PINp});
        ents.push_back({m->fc_embed_w, m->FCXp, H, m->FCXp});
        ents.push_back({m->P("ctx2pool.weight"), H, A, H});
        ents.push_back({m->P("ctx2att.weight"), H, A, H});
        ents.push_back({m->P("att_embed.0.0.weight"), m->rgb, H / 2, m->rgb});
        ents.push_back({m->P("att_embed.1.0.weight"), m->motion, H / 2, m->motion});
        ents.push_back({m->P("core.att_lstm.weight_ih"), H + E, 4 * H, H});                 // pre_att: the fc_feats columns
        ents.push_back({m->P("logit.weight"), H, V, H});
        ents.push_back({m->h2att_w, H, 2 * A, H});
        ents.push_back({m->w_att_cat, H + E, 4 * H, H + E});       // A operands of the conversion-free decode products (skinny_f16_kernel)
        ents.push_back({m->w_lang_cat, 3 * H, 4 * H, 3 * H});
        for (int l = 0; l < 2; ++l) {
            ents.push_back({m->gru_wih[l], l == 0 ? H : 2 * G, 6 * G, l == 0 ? H : 2 * G});
            ents.push_back({m->gru_whh[l], G, 6 * G, G});          // [2 directions][3G][G]: B operand of the tensor-core GRU step
            if (d.obj_interact) {
                const std::string p = "obj_interact.encoder.layers." + std::to_string(l) + ".";
                ents.push_back({m->wqk[l], H, 3 * m->HP, H});
                ents.push_back({m->wo[l], m->HP, H, m->HP});
                ents.push_back({m->P(p + "feedforward.layer.linear1.weight"), H, H / 2, H});
                ents.push_back({m->P(p + "feedforward.layer.linear2.weight"), H / 2, H, H / 2});
            }
        }
        size_t total = 0;
        for (auto& e : ents) total += rup((size_t)e.N * (size_t)((e.K + 31) / 32 * 32), 64);
        if (!m->packed16) GVD_CHECK_CUDA(cudaMalloc(&m->packed16, total * sizeof(float)));
        size_t off = 0;
        std::lock_guard<std::mutex> lk(g_pw_mu);
        for (const float* k : m->pw_keys) g_pw.erase(k);
        m->pw_keys.clear();
        for (auto& e : ents) {
            const long long Kp = (e.K + 31) / 32 * 32;
            GVD_TRY(gvd_pack_f16x3(e.W, e.ldw, e.N, e.K, m->packed16 + off, Kp, st));
            g_pw[e.W] = PackedW{m->packed16 + off, Kp, e.N, e.K, e.ldw};
            m->pw_keys.push_back(e.W);
            off += rup((size_t)e.N * (size_t)Kp, 64);
        }
    }
    m->finalized = true;
    return 0;
}

// ------------------------------------------------------------------------------------ workspace
struct WS {
    // inputs staged for the host-buffer entry point
    float *in_segs, *in_ppls, *in_feat, *out_att2, *out_sim, *out_logp;
    long long *in_num, *in_sidx, *out_seq;
    unsigned char* in_mask;
    // prologue
    float *fc_mean, *xcat, *fc_feats, *g_pool, *simT, *pool_in, *pool_embed, *pool_feats, *tmp_a, *qk, *vT, *vTl, *khi, *klo, *smxF, *S, *att_o, *ffn_h,
        *p_pool, *e, *gi, *gru_out0, *conv, *p_conv, *gh, *hstate;
    // decode
    float *pre_att, *h_att, *c_att, *h_lang, *c_lang, *q, *partial, *x_lang, *logits, *xt;
    float *xcat_att, *xcat_lang, *sk_part;   // split-K path: concatenated LSTM inputs, transposed partial sums [S][B][Nw]
    float *xp_att, *xp_lang;                 // the same concatenated inputs as fp16x3 operand images (conversion-free products, bit 4)
    float* q_part;                           // [4][B][2A] split-K partials of the query projection (summed inside the attention kernel)
    float *k_img, *vt_img;                   // fp16x3 images of the keys (per head) and of V^T for the fused self-attention (bit 8)
    float* a_pk_frame;                       // ... and the frame branch's own (P7 runs on a second stream next to P2-P6)
    float* a_pk;                             // fp16x3 image of the activation operand of the current prologue GEMM (bit 7)
    float *img_h, *img_ffn, *img_g;          // operand images written by the PRODUCER of an activation (GEMM epilogue / row kernel) instead of
                                             // a pack pass: [BR, H] (region embedding / encoder state), [BR, H/2] (FFN hidden), [BR, 2048] (fc7)
    int sk_ldp;
    long long* it;
    unsigned int* gru_bar;             // [2] arrival counters of the persistent GRU layer kernel
    float* h_img;                      // [2 parity][2 dir][B][G] words: fp16x3 images of the GRU state (tensor-core step kernel)
    int* ticket;                       // [rows] last-CTA tickets of the fused attention combine
    float* pk_part; int* pk_ticket;    // fused vocabulary head + greedy pick: per-CTA partials, one ticket
    // beam search (rows = B * beam)
    BeamBufs bb;
    int* bos_att;
    float *z_rows, *gather_tmp;
    // teacher-forced path (MLE / GRD)
    float *ov, *outs, *z_all, *emb, *G, *logits_all, *part_sum;
    unsigned char *labels, *fm;
    int *target, *pred_cls, *cls_idx, *part_cnt;
    long long* tok_col;
    int RC, TC, nch_r, nch_t, clip_chunk, beam, nbox;
    size_t bytes;
};

static void attn_chunking(int B, int R, int T, int* RC, int* TC) {
    const int target = std::max(1, gvd_cdiv(592, B));          // ~4 work items per SM
    auto pick = [&](int n) {
        int c = gvd_cdiv(n, target);
        c = (c + 7) / 8 * 8;
        return std::min(128, std::max(16, c));
    };
    *RC = pick(R);
    *TC = pick(T);
    // measurement aid: rows per region chunk (the CTA count of the decode attention: B * (ceil(R / RC) + ceil(T / TC)) on 2 CTAs per SM)
    if (const char* e = getenv("GVD_ATTN_RC")) { const int v = atoi(e); if (v >= 16 && v <= 128) *RC = (v + 7) / 8 * 8; }
    if (const char* e = getenv("GVD_ATTN_TC")) { const int v = atoi(e); if (v >= 16 && v <= 128) *TC = (v + 7) / 8 * 8; }
}

static WS ws_layout(const gvd_model* m, int B, int T, void* base, int beam = 1, int nbox = 0) {
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, A = d.att_hid_size, R = m->R, G = m->G;
    WS w{};
    size_t off = 0;
    char* b0 = (char*)base;
    auto take = [&](size_t bytes) { size_t o = off; off += rup(bytes, 256); return (void*)(b0 ? b0 + o : (char*)0 + o); };
    const size_t BR = (size_t)B * R, BT = (size_t)B * T;
    const size_t BD = (size_t)B * beam;       // decode rows (beam rows of one clip share its features)
    w.beam = beam;
    attn_chunking((int)BD, R, T, &w.RC, &w.TC);
    gvd_attn_chunks(R, T, w.RC, w.TC, &w.nch_r, &w.nch_t);
    w.clip_chunk = std::max(1, std::min(B, (int)(100000000ll / ((long long)m->nheads * R * R * 4 + 1))));   // S chunk ~<= 100 MB (L2)
    // the attention kernels run one CTA per (clip, head, 128 query rows) and one CTA per SM: a chunk that is one full wave
    // (148 SMs -> 3 clips x 6 heads x 8 row blocks = 144 CTAs at R = 1000) has no partial second wave
    w.clip_chunk = std::max(1, std::min(w.clip_chunk, 148 / std::max(1, m->nheads * ((R + 127) / 128))));
    {
        static const int env_chunk = getenv("GVD_CLIP_CHUNK") ? atoi(getenv("GVD_CLIP_CHUNK")) : 0;
        if (env_chunk > 0) w.clip_chunk = std::min(B, env_chunk);
    }
    w.in_segs = (float*)take(BT * d.fc_feat_size * 4);
    w.in_ppls = (float*)take(BR * 7 * 4);
    w.in_feat = (float*)take(BR * d.att_feat_size * 4);
    w.in_num = (long long*)take((size_t)B * 7 * 8);
    w.in_sidx = (long long*)take((size_t)B * 2 * 8);
    w.in_mask = (unsigned char*)take((size_t)B * (R + 1));
    w.out_seq = (long long*)take((size_t)B * d.seq_length * 8);
    w.out_logp = (float*)take((size_t)B * d.seq_length * 4);
    w.out_att2 = (float*)take((size_t)B * d.seq_length * R * 4);
    w.out_sim = (float*)take((size_t)B * m->NC * R * 4);
    w.fc_mean = (float*)take((size_t)B * d.fc_feat_size * 4);
    w.xcat = (float*)take((size_t)B * m->FCXp * 4);
    w.fc_feats = (float*)take((size_t)B * H * 4);
    w.g_pool = (float*)take(BR * 2048 * 4);
    w.simT = (float*)take(BR * m->NCp * 4);
    w.pool_in = (float*)take(BR * m->PINp * 4);
    w.pool_embed = (float*)take(BR * H * 4);
    if (d.obj_interact) {
        w.pool_feats = (float*)take(BR * H * 4);
        w.tmp_a = (float*)take(BR * H * 4);
        w.qk = (float*)take(BR * 3 * m->HP * 4);
        w.vT = (float*)take((size_t)B * m->HP * R * 4);
        w.vTl = (float*)take((size_t)B * m->HP * R * 4);          // tf32 lo plane of V^T (vT then holds the hi plane)
        w.khi = (float*)take(BR * m->HP * 4);                     // tf32 hi / lo planes of the key projections
        w.klo = (float*)take(BR * m->HP * 4);
        w.smxF = (float*)take((size_t)w.clip_chunk * m->nheads * ((R + 31) / 32) * R * 4);   // softmax group factors of one chunk
        w.S = (float*)take((size_t)w.clip_chunk * m->nheads * R * R * 4);
        w.att_o = (float*)take(BR * m->HP * 4);
        w.k_img = (float*)take(BR * (size_t)m->nheads * ((m->HS + 31) / 32 * 32) * 4);
        w.vt_img = (float*)take((size_t)B * m->HP * ((R + 31) / 32 * 32) * 4);
        w.ffn_h = (float*)take(BR * (H / 2) * 4);
    } else {
        w.pool_feats = w.pool_embed;
    }
    w.p_pool = (float*)take(BR * A * 4);
    w.a_pk = (float*)take(BR * (size_t)std::max(std::max(m->PINp + 32, 2048 + 32), m->HP + 32) * 4);
    w.img_h = (float*)take(BR * (size_t)((m->d.rnn_size + 31) / 32 * 32) * 4);
    w.img_ffn = (float*)take(BR * (size_t)((m->d.rnn_size / 2 + 31) / 32 * 32) * 4);
    w.img_g = (float*)take(BR * (size_t)2048 * 4);
    w.e = (float*)take(BT * H * 4);
    w.gi = (float*)take(BT * 6 * G * 4);
    w.gru_out0 = (float*)take(BT * 2 * G * 4);
    w.conv = (float*)take(BT * H * 4);
    w.p_conv = (float*)take(BT * A * 4);
    w.gh = (float*)take((size_t)2 * B * 3 * G * 4);
    w.hstate = (float*)take((size_t)2 * 2 * B * G * 4);
    w.gru_bar = (unsigned int*)take(256);
    w.h_img = (float*)take((size_t)2 * 2 * B * G * 4);
    w.a_pk_frame = (float*)take(BT * (size_t)((std::max(H, 2 * G) + 31) / 32 * 32 + 32) * 4);   // the frame branch's own pack buffer (it runs concurrently with the region stages)
    w.pre_att = (float*)take((size_t)B * 4 * H * 4);
    w.h_att = (float*)take(2 * BD * H * 4);
    w.c_att = (float*)take(BD * H * 4);
    w.h_lang = (float*)take(2 * BD * H * 4);
    w.c_lang = (float*)take(BD * H * 4);
    w.q = (float*)take(BD * 2 * A * 4);
    w.partial = (float*)take(BD * (w.nch_r + w.nch_t) * (H + 4) * 4);
    w.x_lang = (float*)take(BD * H * 4);
    w.logits = (float*)take(BD * m->Vp * 4);
    w.it = (long long*)take(BD * 8);
    w.xt = (float*)take(BD * d.input_encoding_size * 4);
    w.sk_ldp = (int)rup(BD, 4);
    w.xcat_att = w.xcat_lang = w.sk_part = w.xp_att = w.xp_lang = nullptr;
    if (BD <= 128) {    // operand-swapped split-K path (experimental, backend bit 3): at most 148 (weight-row tile, K split) pairs per product
        w.xcat_att = (float*)take(BD * (size_t)(d.input_encoding_size + H) * 4);
        w.xcat_lang = (float*)take(BD * (size_t)3 * H * 4);
        w.sk_part = (float*)take((size_t)148 * 128 * w.sk_ldp * 4 + (size_t)BD * 64);      // [S][B][ldp], S * ceil(Nw/128) <= 148, ldp <= Nw + 3
        w.xp_att = (float*)take(BD * (size_t)(d.input_encoding_size + H) * 4);
        w.xp_lang = (float*)take(BD * (size_t)3 * H * 4);
        w.q_part = (float*)take((size_t)4 * BD * 2 * A * 4);
    }
    w.ticket = (int*)take(BD * 4);
    w.pk_part = (float*)take((size_t)gvd_cdiv(d.vocab_size, 32) * 128 * 8 * 4);
    w.pk_ticket = (int*)take(256);
    if (beam > 1) {
        const size_t L = d.seq_length, K = beam;
        w.bb.seq = (int*)take((size_t)B * L * K * 4);
        w.bb.att = (int*)take((size_t)B * L * K * 4);
        w.bb.lp = (float*)take((size_t)B * L * K * 4);
        w.bb.sums = (float*)take((size_t)B * K * 4);
        w.bb.parent = (int*)take(BD * 4);
        w.bb.att_ind = (int*)take(BD * 4);
        w.bb.done_flag = (int*)take((size_t)B * 4);
        w.bb.done_slot = (int*)take((size_t)B * 4);
        w.bb.done_seq = (int*)take((size_t)B * L * 4);
        w.bb.done_lp = (float*)take((size_t)B * L * 4);
        w.bb.topv = (float*)take(BD * K * 4);
        w.bb.topi = (int*)take(BD * K * 4);
        w.bb.tokens = (long long*)take(BD * 8);
        w.bos_att = (int*)take(BD * 4);
        w.z_rows = (float*)take(BD * R * 4);
        w.gather_tmp = (float*)take(BD * H * 4);
    }
    w.nbox = nbox;
    if (nbox > 0) {
        const size_t L = d.seq_length, NB = nbox;
        w.ov = (float*)take(BR * NB * 4);
        w.target = (int*)take((size_t)B * NB * R * 4);
        w.pred_cls = (int*)take(BR * 4);
        w.labels = (unsigned char*)take((size_t)B * L * R);
        w.fm = (unsigned char*)take((size_t)B * L * (R + 1));
        w.outs = (float*)take((size_t)B * L * H * 4);
        w.z_all = (float*)take((size_t)B * L * R * 4);
        w.emb = (float*)take((size_t)B * L * 2048 * 4);
        w.cls_idx = (int*)take((size_t)B * L * 4);
        w.G = (float*)take((size_t)B * L * R * 4);
        w.logits_all = (float*)take((size_t)B * L * m->Vp * 4);
        w.part_sum = (float*)take(std::max((size_t)B * L, (size_t)B * NB) * 4);
        w.part_cnt = (int*)take(std::max((size_t)B * L, (size_t)B * NB) * 4);
        w.tok_col = (long long*)take((size_t)B * 8);
    }
    w.bytes = off;
    return w;
}

extern "C" GVD_API size_t gvd_workspace_bytes(const gvd_model_t* m, int B, int T) {
    if (!m || B < 1 || T < 1) return 0;
    return ws_layout(m, B, T, nullptr).bytes;
}
extern "C" GVD_API size_t gvd_workspace_bytes_teacher(const gvd_model_t* m, int B, int T, int nbox) {
    if (!m || B < 1 || T < 1 || nbox < 1) return 0;
    return ws_layout(m, B, T, nullptr, 1, nbox).bytes;
}
extern "C" GVD_API size_t gvd_workspace_bytes_beam(const gvd_model_t* m, int B, int T, int beam_size) {
    if (!m || B < 1 || T < 1 || beam_size < 1) return 0;
    return ws_layout(m, B, T, nullptr, beam_size).bytes;
}

extern "C" GVD_API float* gvd_workspace_tensor(const gvd_model_t* m, void* workspace, int B, int T, const char* name) {
    if (!m || !workspace || !name) return nullptr;
    WS w = ws_layout(m, B, T, workspace);
    const std::string n(name);
    if (n == "fc_feats") return w.fc_feats;
    if (n == "g_pool") return w.g_pool;
    if (n == "pool_embed") return w.pool_embed;
    if (n == "pool_feats") return w.pool_feats;
    if (n == "p_pool_feats") return w.p_pool;
    if (n == "conv_feats") return w.conv;
    if (n == "p_conv_feats") return w.p_conv;
    if (n == "simT") return w.simT;
    if (n == "h_att") return w.h_att;
    if (n == "h_lang") return w.h_lang;
    if (n == "logits") return w.logits;
    return nullptr;
}

static int check_ws(const gvd_model* m, int B, int T, void* workspace, size_t bytes, WS* w, int beam = 1, int nbox = 0) {
    GVD_REQUIRE(m && m->finalized, "model not finalized (call gvd_model_finalize after setting every parameter)");
    GVD_REQUIRE(B >= 1 && T >= 1, "bad batch/frames B=%d T=%d", B, T);
    GVD_REQUIRE(workspace && ((uintptr_t)workspace & 255) == 0, "workspace must be a 256-byte aligned device pointer");
    *w = ws_layout(m, B, T, workspace, beam, nbox);
    GVD_REQUIRE(bytes >= w->bytes, "workspace too small: %zu < %zu bytes", bytes, w->bytes);
    return 0;
}

// ------------------------------------------------------------------------------------ prologue
// C = act(A W^T + bias) for a constant, registered weight W.  Backend bit 7: pack the activation operand into the fp16x3 image (one
// element-wise pass: 4 B read + 4 B written per element) and run the conversion-free kernel (f16ss_kernel: TMA -> tcgen05 SS MMAs);
// otherwise the conversion kernel (tc2_gemm_kernel) on the fp32 operand.
// Pack fusion: the producer of an activation can store its operand image directly (A_img: the image of A, pitch rup32(K), already
// written by whoever produced A; C_img: have THIS GEMM's epilogue store the image of its output, pitch rup32(N)) — the pack pass and
// its 8 B / element of traffic disappear.  C may be null when only the image is consumed.
static bool linear_w_f16ss(const WS& w, const float* W, long long ldw, int M, int N, int K, const float** Wp = nullptr, long long* ldwp = nullptr) {
    const float* p = nullptr;
    long long l = 0;
    const bool ok = (gvd_backend() & 128) != 0 && gvd_gemm_f16() && M >= 1024 && w.a_pk && gvd_packed_lookup(W, ldw, N, K, &p, &l);
    if (Wp) *Wp = p;
    if (ldwp) *ldwp = l;
    return ok;
}
static bool pack_fusion() {
    static const bool off = getenv("GVD_SS_NO_PERSIST") != nullptr;      // (the image is stored by the persistent kernel's epilogue)
    return !off && (gvd_backend() & 512) != 0;                            // backend bit 9
}
static int linear_w(const WS& w, const float* A, long long lda, const float* W, long long ldw, const float* bias, float* C, long long ldc, int M, int N,
                    int K, int act, cudaStream_t st, const float* scale2 = nullptr, const float* shift2 = nullptr, const float* A_img = nullptr,
                    float* C_img = nullptr) {
    const float* Wp = nullptr;
    long long ldwp = 0;
    const long long Kp = (K + 31) / 32 * 32, Np = (N + 31) / 32 * 32;
    if (linear_w_f16ss(w, W, ldw, M, N, K, &Wp, &ldwp)) {
        if (!A_img) {
            GVD_REQUIRE(A, "linear_w: no operand");
            GVD_STAGE("kernel.pack_f16x3", gvd_pack_f16x3(A, lda, M, K, w.a_pk, Kp, st, GVD_F16_SA));
            A_img = w.a_pk;
        }
        GVD_STAGE("kernel.f16ss_gemm", gvd_gemm_f16ss(A_img, Kp, Wp, ldwp, bias, scale2, shift2, act, C, ldc, M, N, K, st, C_img, C_img ? Np : 0));
        return 0;
    }
    GVD_REQUIRE(A && C, "linear_w: the conversion kernel needs the fp32 operand and output");
    GemmArgs g{};
    g.A = A; g.lda = lda; g.W = W; g.ldw = ldw; g.C = C; g.ldc = ldc; g.bias = bias; g.scale2 = scale2; g.shift2 = shift2;
    g.M = M; g.N = N; g.K = K; g.nh = 1; g.act = act; g.alpha = 1.f;
    GVD_TRY(gvd_gemm_nt(g, 1, st));
    if (C_img) GVD_TRY(gvd_pack_f16x3(C, ldc, M, N, C_img, Np, st, GVD_F16_SA));
    return 0;
}

// clips [c0, c0 + B) of the batch the workspace was laid out for (every region buffer is clip-major, so a clip range is a row range)
static int obj_interact_fwd(const gvd_model* m, const WS& w0, int c0, int B, cudaStream_t st, bool fuse) {
    GvdF16Scope f16;
    const int H = m->d.rnn_size, R = m->R, HP = m->HP, HS = m->HS, nh = m->nheads;
    const long long BR = (long long)B * R, r0 = (long long)c0 * R;
    WS w = w0;
    w.pool_embed += r0 * H; w.pool_feats += r0 * H; w.tmp_a += r0 * H; w.qk += r0 * 3 * HP; w.vT += (long long)c0 * HP * R; w.vTl += (long long)c0 * HP * R; w.khi += r0 * HP; w.klo += r0 * HP;
    if (w.k_img) { w.k_img += r0 * nh * ((HS + 31) / 32 * 32); w.vt_img += (long long)c0 * HP * ((R + 31) / 32 * 32); }
    w.att_o += r0 * HP; w.ffn_h += r0 * (H / 2);
    const float* x = w.pool_embed;
    // pack fusion (decided by the caller): w.img_h holds the operand image of x on entry (written by the region-embedding GEMM) and of the
    // encoder state after every add & norm (on exit: of the output); the FFN hidden layer exists only as an image
    for (int l = 0; l < 2; ++l) {
        const std::string p = "obj_interact.encoder.layers." + std::to_string(l) + ".";
        // Q|K|V projections for every region in one GEMM (bias-free, transformer.py:111-114,119)
        const bool fused = (gvd_backend() & 3) == 3 && HS <= 192;
        const bool att16 = fused && (gvd_backend() & 256) != 0 && w.k_img != nullptr;      // fp16x3 images instead of tf32 planes (bit 8)
        const int KH = (HS + 31) / 32 * 32, Rp = (R + 31) / 32 * 32;
        // pack fusion of the attention operands: the projection's epilogue stores Q as fp32, K as the per-head image and V as the image of V^T
        static const bool no_qkv_img = getenv("GVD_NO_QKV_IMG") != nullptr;
        const float* Wp = nullptr;
        long long ldwp = 0;
        const bool qkv_img = fuse && att16 && !no_qkv_img && R % 2 == 0 && HS % 4 == 0 && linear_w_f16ss(w, m->wqk[l], H, (int)BR, 3 * HP, H, &Wp, &ldwp);
        if (qkv_img) {
            GvdQkvImages qi{HP, HS, KH, nh, R, Rp, w.k_img, w.vt_img, GVD_ATT_SK_HOST, GVD_ATT_SV_HOST};
            ProfScope _pk("kernel.f16ss_gemm", st);
            GVD_STAGE("interact.qkv_proj", gvd_gemm_f16ss(w.img_h, (H + 31) / 32 * 32, Wp, ldwp, nullptr, nullptr, nullptr, GVD_ACT_NONE, w.qk, 3 * HP, (int)BR, 3 * HP, H,
                                                          st, nullptr, 0, &qi));
        } else
        GVD_STAGE("interact.qkv_proj", linear_w(w, x, H, m->wqk[l], H, nullptr, w.qk, 3 * HP, (int)BR, 3 * HP, H, GVD_ACT_NONE, st, nullptr, nullptr,
                                                fuse ? w.img_h : nullptr));
        if (qkv_img) {
        } else if (att16) {
            GVD_STAGE("interact.k_split", gvd_pack_heads_f16x3(w.qk + HP, 3 * HP, BR, nh, HS, HS, KH, GVD_ATT_SK_HOST, w.k_img, st));
            GVD_STAGE("interact.v_transpose", gvd_transpose_pack_f16x3(w.qk + 2 * HP, w.vt_img, B, R, HP, 3 * HP, Rp, GVD_ATT_SV_HOST, st));
        } else if (fused) {
            // tf32 hi / lo planes of K and V^T, made once per layer: the two attention kernels then stream them without converting
            GVD_STAGE("interact.k_split", gvd_split_hilo(w.qk + HP, 3 * HP, w.khi, w.klo, HP, BR, HP, st));
            GVD_STAGE("interact.v_transpose", gvd_transpose_split(w.qk + 2 * HP, w.vT, w.vTl, B, R, HP, 3 * HP, st));
        } else {
            // V^T per clip (the P.V product is then again an NT GEMM with K = R contiguous)
            GVD_STAGE("interact.v_transpose", gvd_transpose(w.qk + 2 * HP, w.vT, B, R, HP, 3 * HP, st));
        }
        // The P.V epilogue stores the operand image of the output projection's input (no fp32 att_o, no pack pass).  Through the staged, coalesced
        // epilogue (session 38): P.V 1.98 -> 2.12 ms per step, Wo + pack 1.75 -> 1.30 ms.  (Thread-per-row stores of the image words, session 36:
        // P.V 2.60 ms — slower than the pack pass it removed.)  GVD_NO_ATT_O_IMG restores the pack pass.
        static const bool no_o_img = getenv("GVD_NO_ATT_O_IMG") != nullptr;
        const long long HPi = (HP + 31) / 32 * 32;
        const bool o_img = fuse && att16 && !no_o_img && HS % 4 == 0 && linear_w_f16ss(w, m->wo[l], HP, (int)BR, H, HP);
        for (int b0 = 0; b0 < B; b0 += w.clip_chunk) {
            const int cb = std::min(w.clip_chunk, B - b0);
            {   // S[b,h] = Q_h K_h^T  (heads are zero-padded to HS columns)
                GemmArgs g{};
                g.A = w.qk + (long long)b0 * R * 3 * HP; g.lda = 3 * HP; g.sAb = (long long)R * 3 * HP; g.sAh = HS;
                g.W = g.A + HP; g.ldw = 3 * HP; g.sWb = g.sAb; g.sWh = HS;
                g.C = w.S; g.ldc = R; g.sCb = (long long)nh * R * R; g.sCh = (long long)R * R;
                g.M = R; g.N = R; g.K = HS; g.nh = nh; g.alpha = 1.f;
                if (fused) {
                    // scores + softmax numerator in one sweep: E = exp((s - mu_group)/sqrt(d_model)), group factors -> smxF
                    // (the scale is sqrt(1024)=32, not sqrt(d_head): transformer.py:94,111; quirk Q1)
                    g.W = w.khi + (long long)b0 * R * HP; g.ldw = HP; g.sWb = (long long)R * HP;
                    if (att16) {
                        g.W = w.k_img + (long long)b0 * R * nh * KH; g.ldw = (long long)nh * KH; g.sWb = (long long)R * nh * KH; g.sWh = KH;
                        GVD_STAGE("interact.scores", gvd_attn_scores_tc(g, nullptr, w.smxF, 1.f / sqrtf((float)H), cb * nh, st, 1));
                    } else
                    GVD_STAGE("interact.scores", gvd_attn_scores_tc(g, w.klo + (long long)b0 * R * HP, w.smxF, 1.f / sqrtf((float)H), cb * nh, st));
                } else {
                    GVD_STAGE("interact.scores", gvd_gemm_nt(g, cb * nh, st));
                }
            }
            // softmax(S / sqrt(d_model)) — the scale is sqrt(1024)=32, not sqrt(d_head) (transformer.py:94,111; quirk Q1)
            if (!fused) GVD_STAGE("interact.softmax", gvd_scaled_softmax_rows(w.S, (long long)cb * nh * R, R, R, 1.f / sqrtf((float)H), st));
            {   // O_h = P V_h
                GemmArgs g{};
                g.A = w.S; g.lda = R; g.sAb = (long long)nh * R * R; g.sAh = (long long)R * R;
                g.W = w.vT + (long long)b0 * HP * R; g.ldw = R; g.sWb = (long long)HP * R; g.sWh = (long long)HS * R;
                g.C = w.att_o + (long long)b0 * R * HP; g.ldc = HP; g.sCb = (long long)R * HP; g.sCh = HS;
                g.M = R; g.N = HS; g.K = R; g.nh = nh; g.alpha = 1.f;
                if (att16) {
                    g.W = w.vt_img + (long long)b0 * HP * Rp; g.ldw = Rp; g.sWb = (long long)HP * Rp; g.sWh = (long long)HS * Rp;
                    // pack fusion: the epilogue stores the operand image of the output projection's input (a_pk, free here) instead of fp32 att_o
                    GVD_STAGE("interact.pv", gvd_attn_pv_tc(g, nullptr, w.smxF, cb * nh, st, 1, o_img ? w.a_pk + (long long)b0 * R * HPi : nullptr, HPi));
                } else if (fused) GVD_STAGE("interact.pv", gvd_attn_pv_tc(g, w.vTl + (long long)b0 * HP * R, w.smxF, cb * nh, st));
                else GVD_STAGE("interact.pv", gvd_gemm_nt(g, cb * nh, st));
            }
        }
        GVD_STAGE("interact.wo", linear_w(w, w.att_o, HP, m->wo[l], HP, nullptr, w.tmp_a, H, (int)BR, H, HP, GVD_ACT_NONE, st, nullptr, nullptr, o_img ? w.a_pk : nullptr));
        GVD_STAGE("interact.add_ln", gvd_add_ln_star(x, w.tmp_a, m->P(p + "selfattn.layernorm.gamma"), m->P(p + "selfattn.layernorm.beta"), w.pool_feats, BR, H, st,
                                                     fuse ? w.img_h : nullptr));
        const float* w1 = m->P(p + "feedforward.layer.linear1.weight");
        const float* w2 = m->P(p + "feedforward.layer.linear2.weight");
        const bool hid_img = fuse && linear_w_f16ss(w, w1, H, (int)BR, H / 2, H) && linear_w_f16ss(w, w2, H / 2, (int)BR, H, H / 2);
        GVD_STAGE("interact.ffn1", linear_w(w, w.pool_feats, H, w1, H, m->P(p + "feedforward.layer.linear1.bias"), hid_img ? nullptr : w.ffn_h, H / 2, (int)BR,
                                            H / 2, H, GVD_ACT_RELU, st, nullptr, nullptr, fuse ? w.img_h : nullptr, hid_img ? w.img_ffn : nullptr));
        GVD_STAGE("interact.ffn2", linear_w(w, w.ffn_h, H / 2, w2, H / 2, m->P(p + "feedforward.layer.linear2.bias"), w.tmp_a, H, (int)BR, H, H / 2, GVD_ACT_NONE,
                                            st, nullptr, nullptr, hid_img ? w.img_ffn : nullptr));
        GVD_STAGE("interact.add_ln", gvd_add_ln_star(w.pool_feats, w.tmp_a, m->P(p + "feedforward.layernorm.gamma"), m->P(p + "feedforward.layernorm.beta"),
                                w.pool_feats, BR, H, st, fuse ? w.img_h : nullptr));
        x = w.pool_feats;
    }
    return 0;
}

static int frame_branch_fwd(const gvd_model* m, const WS& w0, int B, int T, const float* segs, const long long* sample_idx,
                            cudaStream_t st) {
    GvdF16Scope f16;
    WS w = w0;
    w.a_pk = w0.a_pk_frame;                 // (the region stages may be packing into a_pk on another stream)
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, A = d.att_hid_size, G = m->G, FC = d.fc_feat_size;
    const long long BT = (long long)B * T;
    // att_embed (rgb | motion) -> BatchNorm1d(eval) -> ReLU fused into the GEMM epilogue (model.py:556-560)
    {
        GemmArgs g{};
        g.A = segs; g.lda = FC; g.W = m->P("att_embed.0.0.weight"); g.ldw = m->rgb; g.bias = m->P("att_embed.0.0.bias");
        g.C = w.e; g.ldc = H; g.M = (int)BT; g.N = H / 2; g.K = m->rgb; g.nh = 1; g.alpha = 1.f;
        g.act = GVD_ACT_RELU_AFFINE_RELU; g.scale2 = m->bn_scale; g.shift2 = m->bn_shift;
        GVD_STAGE("frame.att_embed", gvd_gemm_nt(g, 1, st));
        g.A = segs + m->rgb; g.W = m->P("att_embed.1.0.weight"); g.ldw = m->motion; g.bias = m->P("att_embed.1.0.bias");
        g.C = w.e + H / 2; g.K = m->motion; g.scale2 = m->bn_scale + H / 2; g.shift2 = m->bn_shift + H / 2;
        GVD_STAGE("frame.att_embed", gvd_gemm_nt(g, 1, st));
    }
    // 2-layer bidirectional GRU, hidden G per direction (model.py:150-154,562)
    for (int l = 0; l < 2; ++l) {
        const float* xin = l == 0 ? w.e : w.gru_out0;
        const int in = l == 0 ? H : 2 * G;
        float* out = l == 0 ? w.gru_out0 : w.conv;
        GVD_STAGE("frame.gru_in", linear_w(w, xin, in, m->gru_wih[l], in, m->gru_bih[l], w.gi, 6 * G, (int)BT, 6 * G, in, GVD_ACT_NONE, st));
        if ((gvd_backend() & 32) != 0 && G % 4 == 0 && G <= 1024) {
            // persistent layer kernel: W_hh resident in shared memory, one cooperative launch for all T steps of both directions
            GVD_STAGE("frame.gru_layer", gvd_gru_layer(w.gi, m->gru_whh[l], m->gru_bhh[l], w.hstate, out, l == 1 ? sample_idx : nullptr, w.gru_bar, B, T, G, st));
            continue;
        }
        GVD_CHECK_CUDA(cudaMemsetAsync(w.hstate, 0, (size_t)2 * 2 * B * G * sizeof(float), st));
        {
            // tensor-core step kernel (bit 4): gh = W_hh h on tcgen05 from two pre-split operands with the gate math in the epilogue — one
            // launch per time step instead of a CUDA-core GEMM + a pointwise kernel
            static const bool old_gru = getenv("GVD_GRU_OLD") != nullptr;
            const float* Wimg = nullptr;
            long long ldw = 0;
            if (!old_gru && gvd_gemm_f16() && B <= 128 && G % 32 == 0 && gvd_packed_lookup(m->gru_whh[l], G, 6 * G, G, &Wimg, &ldw)) {
                GVD_STAGE("frame.gru_layer_tc", gvd_gru_layer_f16(w.gi, Wimg, m->gru_bhh[l], w.hstate, w.h_img, out, l == 1 ? sample_idx : nullptr, B, T, G, st));
                continue;
            }
        }
        for (int s = 0; s < T; ++s) {
            float* h_prev = w.hstate + (size_t)(s & 1) * 2 * B * G;
            float* h_new = w.hstate + (size_t)((s + 1) & 1) * 2 * B * G;
            GemmArgs g{};
            g.A = h_prev; g.lda = G; g.sAb = (long long)B * G;
            g.W = m->gru_whh[l]; g.ldw = G; g.sWb = (long long)3 * G * G;
            g.bias = m->gru_bhh[l]; g.sBb = 3 * G;
            g.C = w.gh; g.ldc = 3 * G; g.sCb = (long long)B * 3 * G;
            g.M = B; g.N = 3 * G; g.K = G; g.nh = 1; g.alpha = 1.f;
            GVD_STAGE("frame.gru_hh", gvd_gemm_nt(g, 2, st));
            GVD_STAGE("frame.gru_pointwise", gvd_gru_pointwise(w.gi, w.gh, h_prev, h_new, out, l == 1 ? sample_idx : nullptr, B, T, G, s, st));
        }
    }
    GVD_STAGE("frame.ctx2att", gvd_linear(w.conv, H, m->P("ctx2att.weight"), H, m->P("ctx2att.bias"), w.p_conv, A, (int)BT, A, H, GVD_ACT_NONE, st));
    return 0;
}

// P2-P6 for clips [c0, c0 + cb): per-clip independent, so the host-buffer entry point can run it chunk by chunk
// while the next chunk's fc6 features are still crossing PCIe.  Input pointers are already offset to clip c0.
static int region_prologue(const gvd_model* m, const WS& w0, int c0, int cb, const float* ppls, const float* ppls_feat,
                           const uint8_t* pnt_mask, float* sim_mat_out, cudaStream_t st) {
    GvdF16Scope f16;
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, A = d.att_hid_size, R = m->R;
    const int B = cb;
    const long long BR = (long long)cb * R, r0 = (long long)c0 * R;
    WS w = w0;
    w.g_pool += r0 * 2048; w.simT += r0 * m->NCp; w.pool_in += r0 * m->PINp; w.pool_embed += r0 * H; w.p_pool += r0 * A;
    if (d.obj_interact) w.pool_feats += r0 * H; else w.pool_feats = w.pool_embed;
    // P2 fc7 on every RoI (model.py:512-514)
    // pack fusion (see linear_w): fc7's epilogue also stores the image the similarity GEMM streams; the region-embedding row kernel writes the
    // image of its 2784-wide row and nothing else; the embedding GEMM stores the image the encoder's first projection / ctx2pool stream
    const bool fuse = pack_fusion() && H % 64 == 0 && linear_w_f16ss(w, m->P("ctx2pool.weight"), H, (int)BR, A, H) &&
                      linear_w_f16ss(w, m->pool_embed_w, m->PINp, (int)BR, H, m->PINp) && linear_w_f16ss(w, m->vis_relu, 2048, (int)BR, m->NC, 2048) &&
                      (!d.obj_interact || linear_w_f16ss(w, m->wqk[0], H, (int)BR, 3 * m->HP, H));
    GVD_STAGE("region.fc7", linear_w(w, ppls_feat, d.att_feat_size, m->P("ctx2pool_grd.0.weight"), d.att_feat_size, m->P("ctx2pool_grd.0.bias"), w.g_pool,
                       2048, (int)BR, 2048, d.att_feat_size, GVD_ACT_RELU, st, nullptr, nullptr, nullptr, fuse ? w.img_g : nullptr));
    // P3 region-class similarity, stored region-major: simT[(b,r), c] (model.py:519-535)
    GVD_STAGE("region.sim_gemm", linear_w(w, w.g_pool, 2048, m->vis_relu, 2048, m->P("vis_classifiers_bias"), w.simT, m->NCp, (int)BR, m->NC, 2048, GVD_ACT_NONE, st,
                                          nullptr, nullptr, fuse ? w.img_g : nullptr));
    GVD_STAGE("region.sim_softmax", gvd_sim_softmax(w.simT, pnt_mask, B, R, m->NC, m->NCp, st));
    if (sim_mat_out) GVD_STAGE("region.sim_transpose", gvd_transpose(w.simT, sim_mat_out, B, R, m->NC, m->NCp, st));
    // P4 region embedding (model.py:537-547)
    const int PINi = (m->PINp + 31) / 32 * 32;
    GVD_STAGE("region.pool_in", gvd_pool_in(w.g_pool, ppls, w.simT, m->P("loc_fc.0.weight"), m->P("loc_fc.0.bias"), fuse ? nullptr : w.pool_in, BR, 2048, 300, m->NC,
                                            m->NCp, m->PINp, d.num_sampled_frm, st, fuse ? w.a_pk : nullptr, PINi));
    GVD_STAGE("region.pool_embed", linear_w(w, w.pool_in, m->PINp, m->pool_embed_w, m->PINp, m->P("pool_embed.0.bias"), w.pool_embed, H, (int)BR, H, m->PINp,
                       GVD_ACT_RELU, st, nullptr, nullptr, fuse ? w.a_pk : nullptr, fuse ? w.img_h : nullptr));
    // P5 object interaction (model.py:550-551)
    if (d.obj_interact) GVD_TRY(obj_interact_fwd(m, w0, c0, cb, st, fuse));
    // P6 (model.py:554)
    GVD_STAGE("region.ctx2pool", linear_w(w, w.pool_feats, H, m->P("ctx2pool.weight"), H, m->P("ctx2pool.bias"), w.p_pool, A, (int)BR, A, H, GVD_ACT_NONE, st,
                                          nullptr, nullptr, fuse ? w.img_h : nullptr));
    return 0;
}

// P1 + P7 + the constant part of the attention-LSTM gates: everything that only needs the frame features
static int frame_stages(const gvd_model* m, const WS& w, int B, int T, const float* segs_feat, const long long* num, const long long* sample_idx, cudaStream_t st) {
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, E = d.input_encoding_size, FC = d.fc_feat_size;
    // P1 clip vector (model.py:508-510,548)
    GVD_STAGE("clip.frame_mean", gvd_frame_mean(segs_feat, w.fc_mean, B, T, FC, st));
    GVD_STAGE("clip.vector", gvd_clip_vector(w.fc_mean, num, m->P("seg_info_embed.0.weight"), m->P("seg_info_embed.0.bias"), w.xcat, B, FC, 50, m->FCXp, st));
    GVD_STAGE("clip.fc_embed", gvd_linear(w.xcat, m->FCXp, m->fc_embed_w, m->FCXp, m->P("fc_embed.0.bias"), w.fc_feats, H, B, H, m->FCXp, GVD_ACT_RELU, st));
    // P7 frame branch (model.py:556-565)
    GVD_TRY(frame_branch_fwd(m, w, B, T, segs_feat, sample_idx, st));
    // constant part of the attention-LSTM gates: W_ih[:, :H] fc_feats + b_ih + b_hh (fc_feats is the same at every step)
    GVD_STAGE("decode.pre_att", gvd_linear(w.fc_feats, H, m->P("core.att_lstm.weight_ih"), H + E, m->att_bias_sum, w.pre_att, 4 * H, B, 4 * H, H, GVD_ACT_NONE, st));
    return 0;
}

// The frame stages next to the region stages (P2-P6) instead of behind them: the bi-GRU is 2 * 2 * T dependent launches on 32 SMs (17.7 us
// each: 17 ms at the reference-default T = 480) that nothing else in the prologue depends on.  They run on a second stream;
// while they do, the persistent GEMMs of the region stages launch 32 CTAs fewer (gvd_sm_reserve), otherwise every GRU step would wait
// for a whole GEMM to drain.  Off under the stage profiler (its per-stage times are meant to be serial) or with GVD_NO_FRAME_OVERLAP.
static bool frame_overlap_on() { return g_prof_on.load(std::memory_order_relaxed) == 0 && getenv("GVD_NO_FRAME_OVERLAP") == nullptr; }
static int frame_fork(gvd_model* m, cudaStream_t st) {
    if (!m->frame_stream) {
        int lo = 0, hi = 0;
        GVD_CHECK_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        // default priority: measured (B = 100, T = 480, tools/overlap_diag.py) prologue 38.2 ms serial, 30.5 ms with this stream at the default
        // priority; at the highest priority the programmatically serialized GRU chain holds back every region kernel until it ends (39.0 ms)
        GVD_CHECK_CUDA(cudaStreamCreateWithPriority(&m->frame_stream, cudaStreamNonBlocking, getenv("GVD_FRAME_PRIO_HIGH") ? hi : lo));
        GVD_CHECK_CUDA(cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming));
        GVD_CHECK_CUDA(cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming));
    }
    GVD_CHECK_CUDA(cudaEventRecord(m->ev_fork, st));              // the workspace may still be in use by earlier work on `st`
    GVD_CHECK_CUDA(cudaStreamWaitEvent(m->frame_stream, m->ev_fork, 0));
    return 0;
}
static int frame_join(gvd_model* m, cudaStream_t st) {
    GVD_CHECK_CUDA(cudaEventRecord(m->ev_join, m->frame_stream));
    GVD_CHECK_CUDA(cudaStreamWaitEvent(st, m->ev_join, 0));
    return 0;
}
// Clips of the region stages that run with the SM reserve: about as many as the GRU chain lasts (measured: 17.7 us per GRU step, 0.21 ms per
// clip of region stages on 148 SMs), whole attention sub-batches; short clips (T < 64: chain < 2.3 ms) run without a reserve.
// (one GRU step = 2 directions x G / 32 CTAs, one per SM; GVD_FRAME_RESERVE_SMS overrides — more leaves room for the next step's CTAs, which
// programmatic stream serialization schedules early to prefetch their W_hh tiles)
static int frame_reserve_sms(const gvd_model* m) {
    const char* e = getenv("GVD_FRAME_RESERVE_SMS");
    return e ? std::max(0, std::min(120, atoi(e))) : 2 * (m->G / 32);
}
static int frame_reserve_clips(const gvd_model* m, const WS& w, int B, int T) {
    if (T < 64) return 0;
    const double gru_ms = 2.0 * T * 0.0177 + 0.3, clip_ms = 0.21 * 148.0 / (148.0 - frame_reserve_sms(m));
    const double scale = getenv("GVD_FRAME_RESERVE_SCALE") ? atof(getenv("GVD_FRAME_RESERVE_SCALE")) : 1.0;
    if (frame_reserve_sms(m) == 0 || scale <= 0.0) return 0;
    const int n = (int)(scale * gru_ms / clip_ms) + 1;
    return std::min(B, (n + w.clip_chunk - 1) / w.clip_chunk * w.clip_chunk);
}
struct SmReserveScope {
    int old;
    explicit SmReserveScope(int n) : old(gvd_sm_reserve(n)) {}
    ~SmReserveScope() { gvd_sm_reserve(old); }
};

extern "C" GVD_API int gvd_prologue_fwd(gvd_model_t* m, int B, int T, const float* segs_feat, const float* ppls, const int64_t* num,
                                const float* ppls_feat, const int64_t* sample_idx, const uint8_t* pnt_mask, void* workspace,
                                size_t workspace_bytes, float* sim_mat_out, void* stream) {
    WS w;
    GVD_TRY(check_ws(m, B, T, workspace, workspace_bytes, &w));
    GVD_REQUIRE(segs_feat && ppls && num && ppls_feat && sample_idx && pnt_mask, "prologue: null input");
    cudaStream_t st = (cudaStream_t)stream;
    const gvd_dims_t& d = m->d;
    const int R = m->R;
    const bool overlap = frame_overlap_on();
    cudaStream_t fst = st;
    // GVD_TRACE_OVERLAP: when did each stream finish (ms after the fork)?  Diagnostic only: synchronises the stream.
    const bool otrace = overlap && getenv("GVD_TRACE_OVERLAP") != nullptr;
    cudaEvent_t te[3] = {nullptr, nullptr, nullptr};
    if (otrace) for (auto& e : te) GVD_CHECK_CUDA(cudaEventCreate(&e));
    if (overlap) { GVD_TRY(frame_fork(m, st)); fst = m->frame_stream; }
    if (otrace) GVD_CHECK_CUDA(cudaEventRecord(te[0], st));
    const int rc_frame = frame_stages(m, w, B, T, segs_feat, (const long long*)num, (const long long*)sample_idx, fst);
    if (otrace) GVD_CHECK_CUDA(cudaEventRecord(te[1], fst));
    if (overlap && rc_frame != 0) frame_join(m, st);            // never leave the second stream dangling behind an error return
    if (rc_frame != 0) return rc_frame;
    int rc = 0;
    if (getenv("GVD_CHUNKED")) {          // measurement aid: the chunked schedule of the host-buffer entry point, without the copies
        const int chunk = std::max(1, std::min(B, atoi(getenv("GVD_CHUNKED"))));
        for (int c0 = 0; c0 < B && rc == 0; c0 += chunk) {
            const int cb = std::min(chunk, B - c0);
            rc = region_prologue(m, w, c0, cb, ppls + (size_t)c0 * R * 7, ppls_feat + (size_t)c0 * R * d.att_feat_size, pnt_mask + (size_t)c0 * (R + 1),
                                 sim_mat_out ? sim_mat_out + (size_t)c0 * m->NC * R : nullptr, st);
        }
    } else {
        // P2-P6: the first n_res clips next to the GRU chain with the SM reserve, the rest on the whole GPU
        const int n_res = overlap ? frame_reserve_clips(m, w, B, T) : 0;
        if (n_res > 0) {
            SmReserveScope rs(frame_reserve_sms(m));
            rc = region_prologue(m, w, 0, n_res, ppls, ppls_feat, pnt_mask, sim_mat_out, st);
        }
        if (rc == 0 && n_res < B)
            rc = region_prologue(m, w, n_res, B - n_res, ppls + (size_t)n_res * R * 7, ppls_feat + (size_t)n_res * R * d.att_feat_size,
                                 pnt_mask + (size_t)n_res * (R + 1), sim_mat_out ? sim_mat_out + (size_t)n_res * m->NC * R : nullptr, st);
    }
    if (otrace) GVD_CHECK_CUDA(cudaEventRecord(te[2], st));
    if (overlap) GVD_TRY(frame_join(m, st));
    if (otrace) {
        GVD_CHECK_CUDA(cudaStreamSynchronize(st));
        float a = 0.f, b = 0.f;
        cudaEventElapsedTime(&a, te[0], te[1]);
        cudaEventElapsedTime(&b, te[0], te[2]);
        fprintf(stderr, "[gvd] overlap trace: frame stream done %.2f ms, region stages done %.2f ms after the fork (reserve %d SMs for %d clips)\n", a, b,
                frame_reserve_sms(m), frame_reserve_clips(m, w, B, T));
        for (auto& e : te) cudaEventDestroy(e);
    }
    return rc;
}

// ------------------------------------------------------------------------------------ decode
extern "C" GVD_API int gvd_decode_reset_state(gvd_model_t* m, int B, int T, void* workspace, size_t workspace_bytes, void* stream) {
    WS w;
    GVD_TRY(check_ws(m, B, T, workspace, workspace_bytes, &w));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)B * w.beam * m->d.rnn_size * sizeof(float);
    GVD_CHECK_CUDA(cudaMemsetAsync(w.h_att, 0, 2 * n, st));     // init_hidden: zeros (model.py:237-240)
    GVD_CHECK_CUDA(cudaMemsetAsync(w.c_att, 0, n, st));
    GVD_CHECK_CUDA(cudaMemsetAsync(w.h_lang, 0, 2 * n, st));
    GVD_CHECK_CUDA(cudaMemsetAsync(w.c_lang, 0, n, st));
    GVD_CHECK_CUDA(cudaMemsetAsync(w.ticket, 0, (size_t)B * w.beam * sizeof(int), st));
    GVD_CHECK_CUDA(cudaMemsetAsync(w.pk_ticket, 0, sizeof(int), st));
    if (w.xcat_att) {      // split-K path: the recurrent states also live inside the concatenated LSTM inputs
        GVD_CHECK_CUDA(cudaMemsetAsync(w.xcat_att, 0, (size_t)B * w.beam * (m->d.input_encoding_size + m->d.rnn_size) * sizeof(float), st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.xcat_lang, 0, (size_t)B * w.beam * 3 * m->d.rnn_size * sizeof(float), st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.xp_att, 0, (size_t)B * w.beam * (m->d.input_encoding_size + m->d.rnn_size) * sizeof(float), st));   // +0 halves
        GVD_CHECK_CUDA(cudaMemsetAsync(w.xp_lang, 0, (size_t)B * w.beam * 3 * m->d.rnn_size * sizeof(float), st));
    }
    return 0;
}

// does the core step run its three products operand-swapped + split along K (gvd_skinny.cu)?  Then xt / h_att / h_lang live inside the
// concatenated LSTM inputs xcat_att = [xt | h_att] and xcat_lang = [att + att2 | h_att | h_lang].
static bool core_skinny(const gvd_model* m, const WS& w, int B, int div) {
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, A = d.att_hid_size, E = d.input_encoding_size;
    return (gvd_backend() & 1) != 0 && H % 8 == 0 && (gvd_backend() & 8) != 0 && div == 1 && w.sk_part != nullptr && E % 4 == 0 &&
           gvd_skinny_splits(4 * H, E + H, B) > 0 && gvd_skinny_splits(2 * A, H, B) > 0 && gvd_skinny_splits(4 * H, 3 * H, B) > 0;
}

// ... and with backend bit 4 through the conversion-free kernel: weights AND activations in the fp16x3 operand image (needs 32-column
// granularity of every concatenated segment)
static bool core_skinny_f16(const gvd_model* m) {
    const gvd_dims_t& d = m->d;
    return (gvd_backend() & 16) != 0 && d.rnn_size % 32 == 0 && d.input_encoding_size % 32 == 0 && d.att_hid_size % 16 == 0;
}

// B = decode rows (clips x beam); rows [k*div, (k+1)*div) attend over clip k's features / masks
static int core_step(const gvd_model* m, const WS& w, int B, int T, int step, const long long* tokens, const unsigned char* att_mask,
                     const unsigned char* out_mask, float* z_out, long long z_stride_b, cudaStream_t st, int div = 1, long long out_mask_stride = 0,
                     bool xt_ready = false) {
    GvdF16Scope f16;
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, A = d.att_hid_size, E = d.input_encoding_size, R = m->R;
    const size_t BH = (size_t)B * H;
    float* h_att_cur = w.h_att + (size_t)(step & 1) * BH;
    float* h_att_nxt = w.h_att + (size_t)((step + 1) & 1) * BH;
    float* h_lang_cur = w.h_lang + (size_t)(step & 1) * BH;
    float* h_lang_nxt = w.h_lang + (size_t)((step + 1) & 1) * BH;
    const bool tc = (gvd_backend() & 1) != 0 && H % 8 == 0;
    // operand-swapped split-K products (gvd_skinny.cu): experimental, backend bit 3; one `pre` row per batch row only
    const bool skinny = core_skinny(m, w, B, div);
    const bool sk16 = skinny && core_skinny_f16(m);     // both operands pre-split: conversion-free products (skinny_f16_kernel)
    {   // attention LSTM: input cat(fc_feats, xt), xt = ReLU(embed[token]) (AttModel.py:138-139)
        LstmArgs a{};
        a.nseg = 2;
        a.seg[0] = LstmSeg{m->P("embed.0.weight"), E, tokens, 1, m->P("core.att_lstm.weight_ih") + H, H + E, E};
        a.seg[1] = LstmSeg{h_att_cur, H, nullptr, 0, m->P("core.att_lstm.weight_hh"), H, H};
        a.pre = w.pre_att; a.pre_div = div;
        a.c_prev = w.c_att; a.c_out = w.c_att; a.h_out = h_att_nxt; a.B = B; a.H = H;
        if (tc) {
            // split-K path: the input [xt | h_att(t-1)] is ONE matrix (xcat_att): the sampler / this embedding write xt into its first E
            // columns, the previous step's reduction wrote h_att into the rest; no concat launch
            if (!xt_ready) {
                embed_relu_kernel<<<gvd_cdiv((long long)B * E, 256), 256, 0, st>>>(m->P("embed.0.weight"), tokens, skinny ? w.xcat_att : w.xt, skinny ? E + H : E, B,
                                                                                 E, d.vocab_size, sk16 ? w.xp_att : nullptr, E + H);
                GVD_CHECK_LAUNCH();
            }
            a.seg[0] = LstmSeg{w.xt, E, nullptr, 0, m->P("core.att_lstm.weight_ih") + H, H + E, E};
            if (skinny) {
                const int S = gvd_skinny_splits(4 * H, E + H, B);
                const float* Wp; long long ldwp;
                if (sk16 && gvd_packed_lookup(m->w_att_cat, E + H, 4 * H, E + H, &Wp, &ldwp)) {
                    GVD_STAGE("decode.lstm_att", gvd_skinny_f16(Wp, ldwp, 4 * H, w.xp_att, E + H, B, E + H, S, w.sk_part, 4 * H, st));
                } else {
                    GVD_REQUIRE(!sk16, "core_step: packed attention-LSTM weights missing");
                    GVD_STAGE("decode.lstm_att", gvd_skinny_splitk(m->w_att_cat, 4 * H, E + H, w.xcat_att, E + H, B, S, w.sk_part, 4 * H, st));
                }
                GVD_STAGE("decode.lstm_att_reduce", gvd_reduce_lstm(w.sk_part, S, 4 * H, a.pre, a.pre_div, nullptr, nullptr, a.c_prev, a.c_out, a.h_out, H,
                                                                    w.xcat_att + E, E + H, w.xcat_lang + H, 3 * H, B, H, st,
                                                                    sk16 ? w.xp_att + E : nullptr, E + H, sk16 ? w.xp_lang + H : nullptr, 3 * H));
            } else {
                GVD_STAGE("decode.lstm_att", gvd_lstm_step_tc(a, st));
            }
        } else {
            GVD_STAGE("decode.lstm_att", gvd_lstm_step(a, st));
        }
    }
    // both attention queries in one GEMM: q = [h2att(h_a) | h2att2(h_a)]
    int q_S = 0;          // > 0: the queries stay as q_S split-K partials in w.q_part, summed by the attention kernel
    {
        if (skinny) {
            const int S = gvd_skinny_splits(2 * A, H, B);
            const float* Wp; long long ldwp;
            if (sk16 && gvd_packed_lookup(m->h2att_w, H, 2 * A, H, &Wp, &ldwp)) {
                // 4 splits only: the attention kernel sums the partials itself while it loads its query (no reduction launch)
                q_S = std::min(S, 4);
                while (H % (32 * q_S) != 0) --q_S;
                GVD_STAGE("decode.h2att", gvd_skinny_f16(Wp, ldwp, 2 * A, w.xp_lang + H, 3 * H, B, H, q_S, w.q_part, 2 * A, st));       // X = h_att(t) inside xp_lang
            } else {
                GVD_REQUIRE(!sk16, "core_step: packed query weights missing");
                GVD_STAGE("decode.h2att", gvd_skinny_splitk(m->h2att_w, 2 * A, H, h_att_nxt, H, B, S, w.sk_part, 2 * A, st));
            }
            if (!q_S) GVD_STAGE("decode.h2att_reduce", gvd_reduce_bias(w.sk_part, S, 2 * A, 2 * A, m->h2att_b, w.q, 2 * A, B, st));
        } else {
            GVD_STAGE("decode.h2att", gvd_linear(h_att_nxt, H, m->h2att_w, H, m->h2att_b, w.q, 2 * A, B, 2 * A, H, GVD_ACT_NONE, st));
        }
    }
    {
        AttnArgs a{};
        a.p_pool = w.p_pool; a.pool = w.pool_feats; a.p_conv = w.p_conv; a.conv = w.conv; a.q = w.q;
        if (q_S) { a.q = nullptr; a.q_part = w.q_part; a.q_S = q_S; a.q_plane = (long long)B * 2 * A; a.q_bias = m->h2att_b; }
        a.w1 = m->P("core.attention.alpha_net.weight"); a.b1 = m->P("core.attention.alpha_net.bias");
        a.w2 = m->P("core.attention2.alpha_net.weight"); a.b2 = m->P("core.attention2.alpha_net.bias");
        a.att_mask = att_mask; a.out_mask = out_mask; a.z_out = z_out; a.z_stride_b = z_stride_b;
        a.partial = w.partial; a.B = B; a.R = R; a.T = T; a.A = A; a.H = H; a.RC = w.RC; a.TC = w.TC; a.feat_div = div;
        a.out_mask_stride = out_mask_stride;
        a.ticket = w.ticket; a.x_out = w.x_lang;         // chunk partials are merged by the last CTA of each row (no combine launch)
        if (skinny) { a.x_out = w.xcat_lang; a.x_ld = 3 * H; }   // ... straight into the language LSTM's concatenated input
        if (sk16) { a.x_pk = w.xp_lang; a.x_pk_ld = 3 * H; }
        GVD_STAGE("decode.attn_partial", gvd_attn_partial(a, st));
    }
    {   // language LSTM: input cat(att + att2, h_att) (AttModel.py:147-160)
        LstmArgs a{};
        a.nseg = 3;
        a.seg[0] = LstmSeg{w.x_lang, H, nullptr, 0, m->P("core.lang_lstm.weight_ih"), 2 * H, H};
        a.seg[1] = LstmSeg{h_att_nxt, H, nullptr, 0, m->P("core.lang_lstm.weight_ih") + H, 2 * H, H};
        a.seg[2] = LstmSeg{h_lang_cur, H, nullptr, 0, m->P("core.lang_lstm.weight_hh"), H, H};
        a.bias1 = m->P("core.lang_lstm.bias_ih"); a.bias2 = m->P("core.lang_lstm.bias_hh");
        a.c_prev = w.c_lang; a.c_out = w.c_lang; a.h_out = h_lang_nxt; a.B = B; a.H = H;
        if (skinny) {
            const int S = gvd_skinny_splits(4 * H, 3 * H, B);
            const float* Wp; long long ldwp;
            if (sk16 && gvd_packed_lookup(m->w_lang_cat, 3 * H, 4 * H, 3 * H, &Wp, &ldwp)) {
                GVD_STAGE("decode.lstm_lang", gvd_skinny_f16(Wp, ldwp, 4 * H, w.xp_lang, 3 * H, B, 3 * H, S, w.sk_part, 4 * H, st));
            } else {
                GVD_REQUIRE(!sk16, "core_step: packed language-LSTM weights missing");
                GVD_STAGE("decode.lstm_lang", gvd_skinny_splitk(m->w_lang_cat, 4 * H, 3 * H, w.xcat_lang, 3 * H, B, S, w.sk_part, 4 * H, st));
            }
            GVD_STAGE("decode.lstm_lang_reduce", gvd_reduce_lstm(w.sk_part, S, 4 * H, nullptr, 0, a.bias1, a.bias2, a.c_prev, a.c_out, a.h_out, H,
                                                                 w.xcat_lang + 2 * H, 3 * H, nullptr, 0, B, H, st, sk16 ? w.xp_lang + 2 * H : nullptr, 3 * H,
                                                                 nullptr, 0));
        } else if (tc) GVD_STAGE("decode.lstm_lang", gvd_lstm_step_tc(a, st));
        else GVD_STAGE("decode.lstm_lang", gvd_lstm_step(a, st));
    }
    return 0;
}

extern "C" GVD_API int gvd_decode_step_fwd(gvd_model_t* m, int B, int T, void* workspace, size_t workspace_bytes, int step,
                                   const int64_t* tokens, const uint8_t* att_mask, const uint8_t* out_mask, float* att2_logits_out,
                                   int64_t att2_stride_b, float* h_lang_out, void* stream) {
    WS w;
    GVD_TRY(check_ws(m, B, T, workspace, workspace_bytes, &w));
    GVD_REQUIRE(tokens && att_mask && out_mask && att2_logits_out && step >= 0, "decode_step: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    GVD_TRY(core_step(m, w, B, T, step, (const long long*)tokens, att_mask, out_mask, att2_logits_out, att2_stride_b, st));
    if (h_lang_out) {
        const size_t BH = (size_t)B * m->d.rnn_size;
        GVD_CHECK_CUDA(cudaMemcpyAsync(h_lang_out, w.h_lang + (size_t)((step + 1) & 1) * BH, BH * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

// S1: the 21-iteration greedy loop (model.py:579-624) enqueued on `st`; every pointer is fixed for a given workspace, so the
// whole enqueue is capturable as a CUDA graph.
static int decode_greedy_enqueue(gvd_model_t* m, const WS& w, int B, int T, void* workspace, size_t workspace_bytes, const uint8_t* pnt_mask,
                                 int64_t* seq_out, float* logprobs_out, float* att2_logits_out, cudaStream_t st) {
    GvdF16Scope f16;
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, V = d.vocab_size, L = d.seq_length, R = m->R;
    GVD_TRY(gvd_decode_reset_state(m, B, T, workspace, workspace_bytes, (void*)st));
    GVD_CHECK_CUDA(cudaMemsetAsync(w.it, 0, (size_t)B * sizeof(long long), st));            // <bos> = 0 (model.py:587-588)
    // The pick kernel also writes the next step's xt = ReLU(embed[token]) (no separate embedding launch).  Folding the whole
    // sampler into the vocabulary-head GEMM epilogue (mode 2 of tc2_gemm_kernel, last-CTA merge of 154 per-CTA partials) is
    // implemented and parity-tested but measured SLOWER (168 us vs 62 us per step: the merge is a serial chain on one CTA),
    // so it is only used when GVD_FUSED_PICK is set.
    const bool tc = (gvd_backend() & 1) != 0 && H % 8 == 0;
    static const bool fused_pick = getenv("GVD_FUSED_PICK") != nullptr;
    const bool fused = tc && fused_pick && B <= 128;
    for (int t = 0; t < L; ++t) {
        GVD_TRY(core_step(m, w, B, T, t, w.it, pnt_mask, pnt_mask, att2_logits_out + (size_t)t * R, (long long)L * R, st, 1, 0, tc && t > 0));
        const float* h = w.h_lang + (size_t)((t + 1) & 1) * B * H;
        if (fused) {
            GVD_STAGE("decode.logit_pick", gvd_logit_pick_tc(h, H, m->P("logit.weight"), H, m->P("logit.bias"), B, V, H, d.unk_idx, w.pk_part,
                                                             w.pk_ticket, w.it, (long long*)seq_out + t, logprobs_out ? logprobs_out + t : nullptr, L,
                                                             m->P("embed.0.weight"), w.xt, d.input_encoding_size, st));
        } else {
            const int E = d.input_encoding_size;
            const int S = (tc && (gvd_backend() & 8) != 0 && w.sk_part && V <= 6144) ? gvd_skinny_splits(V, H, B) : 0;
            const bool sk_core = core_skinny(m, w, B, 1);                       // then xt goes into the core step's concatenated input
            if (S > 0) {
                // vocabulary head: split-K partials, then ONE kernel sums them, adds the bias and samples (no [B,V] logits round trip)
                const bool sk16 = sk_core && core_skinny_f16(m);
                const float* Wp; long long ldwp;
                if (sk16 && gvd_packed_lookup(m->P("logit.weight"), H, V, H, &Wp, &ldwp)) {
                    GVD_STAGE("decode.logit", gvd_skinny_f16(Wp, ldwp, V, w.xp_lang + 2 * H, 3 * H, B, H, S, w.sk_part, m->Vp, st));     // X = h_lang(t) inside xp_lang
                } else {
                    GVD_REQUIRE(!sk16, "decode: packed vocabulary-head weights missing");
                    GVD_STAGE("decode.logit", gvd_skinny_splitk(m->P("logit.weight"), V, H, h, H, B, S, w.sk_part, m->Vp, st));
                }
                GVD_STAGE("decode.pick", gvd_reduce_pick(w.sk_part, S, m->Vp, m->P("logit.bias"), B, V, d.unk_idx, w.it, (long long*)seq_out + t,
                                                         logprobs_out ? logprobs_out + t : nullptr, L, m->P("embed.0.weight"), sk_core ? w.xcat_att : w.xt,
                                                         sk_core ? E + H : E, E, nullptr, 0, st, sk16 ? w.xp_att : nullptr, E + H));
            } else {
                GVD_STAGE("decode.logit", gvd_linear(h, H, m->P("logit.weight"), H, m->P("logit.bias"), w.logits, m->Vp, B, V, H, GVD_ACT_NONE, st));
                GVD_STAGE("decode.pick", gvd_greedy_pick(w.logits, m->Vp, B, V, d.unk_idx, w.it, (long long*)seq_out + t, logprobs_out ? logprobs_out + t : nullptr,
                                                         L, tc ? m->P("embed.0.weight") : nullptr, tc ? (sk_core ? w.xcat_att : w.xt) : nullptr, E, st, sk_core ? E + H : E));
            }
        }
    }
    return 0;
}

extern "C" GVD_API int gvd_decode_greedy(gvd_model_t* m, int B, int T, void* workspace, size_t workspace_bytes, const uint8_t* pnt_mask,
                                 int64_t* seq_out, float* logprobs_out, float* att2_logits_out, void* stream) {
    WS w;
    GVD_TRY(check_ws(m, B, T, workspace, workspace_bytes, &w));
    GVD_REQUIRE(pnt_mask && seq_out && att2_logits_out, "decode_greedy: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int L = m->d.seq_length, R = m->R;
    // Direct enqueue when the stage profiler is on (its events cannot be captured) or when asked (GVD_NO_GRAPH: per-kernel ncu runs)
    static const bool no_graph = getenv("GVD_NO_GRAPH") != nullptr;
    if (no_graph || g_prof_on.load(std::memory_order_relaxed) != 0)
        return decode_greedy_enqueue(m, w, B, T, workspace, workspace_bytes, pnt_mask, seq_out, logprobs_out, att2_logits_out, st);
    // Graph path: the loop reads the mask from / writes its results to workspace-resident buffers (fixed addresses), the caller's
    // tensors are copied in / out around the replay.
    if (!m->greedy_exec || m->greedy_key.B != B || m->greedy_key.T != T || m->greedy_key.backend != gvd_backend() || m->greedy_key.ws != workspace ||
        m->greedy_key.ws_bytes != workspace_bytes) {
        if (m->greedy_exec) { cudaGraphExecDestroy(m->greedy_exec); m->greedy_exec = nullptr; }
        if (!m->capture_stream) GVD_CHECK_CUDA(cudaStreamCreateWithFlags(&m->capture_stream, cudaStreamNonBlocking));
        cudaGraph_t graph = nullptr;
        GVD_CHECK_CUDA(cudaStreamBeginCapture(m->capture_stream, cudaStreamCaptureModeThreadLocal));
        const long long l0 = g_launches.load();
        const int rc = decode_greedy_enqueue(m, w, B, T, workspace, workspace_bytes, w.in_mask, (int64_t*)w.out_seq, w.out_logp, w.out_att2, m->capture_stream);
        const cudaError_t ce = cudaStreamEndCapture(m->capture_stream, &graph);
        m->greedy_nodes = g_launches.load() - l0;
        g_launches.store(l0);                              // capturing launches nothing
        if (rc != 0) { if (graph) cudaGraphDestroy(graph); return rc; }
        GVD_CHECK_CUDA(ce);
        const cudaError_t ie = cudaGraphInstantiate(&m->greedy_exec, graph, 0);
        cudaGraphDestroy(graph);
        GVD_CHECK_CUDA(ie);
        m->greedy_key = {B, T, gvd_backend(), workspace, workspace_bytes};
    }
    if (pnt_mask != w.in_mask) GVD_CHECK_CUDA(cudaMemcpyAsync(w.in_mask, pnt_mask, (size_t)B * (R + 1), cudaMemcpyDeviceToDevice, st));
    GVD_CHECK_CUDA(cudaGraphLaunch(m->greedy_exec, st));
    g_launches.fetch_add(m->greedy_nodes, std::memory_order_relaxed);
    if (seq_out != (int64_t*)w.out_seq) GVD_CHECK_CUDA(cudaMemcpyAsync(seq_out, w.out_seq, (size_t)B * L * 8, cudaMemcpyDeviceToDevice, st));
    if (logprobs_out && logprobs_out != w.out_logp) GVD_CHECK_CUDA(cudaMemcpyAsync(logprobs_out, w.out_logp, (size_t)B * L * 4, cudaMemcpyDeviceToDevice, st));
    if (att2_logits_out != w.out_att2) GVD_CHECK_CUDA(cudaMemcpyAsync(att2_logits_out, w.out_att2, (size_t)B * L * R * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}

namespace {
__global__ void copy_token_column_kernel(const long long* seq, long long* out, int B, int L1, int i) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) out[b] = seq[(long long)b * L1 + i];
}
}  // namespace

// T1-T6 / G1: teacher-forced forward (misc/model.py:283-489), eval-mode arithmetic.  mode 0 = 'MLE' (four losses),
// mode 1 = 'GRD' (per-frame argmax of attention and grounding logits + region-class predictions).
extern "C" GVD_API int gvd_teacher_fwd(gvd_model_t* m, int B, int T, int nbox, int S, int mode, void* workspace, size_t workspace_bytes,
                                       const int64_t* seq, const int64_t* input_cls, const float* ppls, const float* gt_boxes,
                                       const uint8_t* mask_boxes, const uint8_t* frm_mask, const uint8_t* pnt_mask, float* losses_out,
                                       int64_t* att_idx_out, int64_t* grd_idx_out, int32_t* sim_target_out, int32_t* cls_pred_out, void* stream) {
    WS w;
    GVD_TRY(check_ws(m, B, T, workspace, workspace_bytes, &w, 1, nbox));
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, V = d.vocab_size, L = d.seq_length, R = m->R, L1 = L + 1;
    GVD_REQUIRE(seq && input_cls && ppls && gt_boxes && frm_mask && pnt_mask, "teacher_fwd: null input");
    GVD_REQUIRE(S >= 1 && S <= L && nbox >= 1, "teacher_fwd: need 1 <= S <= seq_length and nbox >= 1 (S=%d nbox=%d)", S, nbox);
    GVD_REQUIRE(mode == 1 || (mask_boxes && losses_out), "teacher_fwd: MLE needs mask_boxes and losses_out");
    GVD_REQUIRE(mode == 0 || (att_idx_out && grd_idx_out), "teacher_fwd: GRD needs the index outputs");
    cudaStream_t st = (cudaStream_t)stream;
    // IoU of every proposal with every GT box, frame + proposal masks applied (model.py:317-318)
    GVD_STAGE("teacher.iou", gvd_bbox_overlaps(ppls, gt_boxes, frm_mask, pnt_mask, w.ov, B, R, nbox, st));
    GVD_STAGE("teacher.cls", gvd_cls_target(w.ov, gt_boxes, w.simT, w.target, w.part_sum, w.part_cnt, B, R, nbox, m->NC, m->NCp, st));
    if (mode == 0) {
        GVD_STAGE("teacher.reduce", gvd_finish_mean(w.part_sum, w.part_cnt, B * nbox, -1.f, losses_out + 3, st));     // cls_loss (model.py:348-350)
        GVD_STAGE("teacher.targets", gvd_step_targets(w.ov, mask_boxes, frm_mask, pnt_mask, w.labels, w.fm, B, S, R, nbox, L1, st));
    } else {
        if (sim_target_out) GVD_CHECK_CUDA(cudaMemcpyAsync(sim_target_out, w.target, (size_t)B * nbox * R * 4, cudaMemcpyDeviceToDevice, st));
        if (cls_pred_out) GVD_STAGE("teacher.cls", gvd_class_argmax(w.simT, (int*)cls_pred_out, (long long)B * R, m->NC, m->NCp, st));
    }
    // teacher-forced loop: step i feeds seq[:, i] (model.py:421-453); S is the reference's early-exit count
    GVD_TRY(gvd_decode_reset_state(m, B, T, workspace, workspace_bytes, stream));
    for (int i = 0; i < S; ++i) {
        copy_token_column_kernel<<<gvd_cdiv(B, 128), 128, 0, st>>>((const long long*)seq, w.tok_col, B, L1, i);
        GVD_CHECK_LAUNCH();
        // MLE: softmax mask = proposal mask, returned logits additionally masked with the step's frame mask (model.py:441-443);
        // GRD: both are the proposal mask (model.py:446-448)
        const unsigned char* out_mask = mode == 0 ? w.fm + (size_t)i * (R + 1) : pnt_mask;
        const long long out_stride = mode == 0 ? (long long)S * (R + 1) : (long long)(R + 1);
        GVD_TRY(core_step(m, w, B, T, i, w.tok_col, pnt_mask, out_mask, w.z_all + (size_t)i * R, (long long)S * R, st, 1, out_stride));
        const float* h = w.h_lang + (size_t)((i + 1) & 1) * B * H;
        GVD_CHECK_CUDA(cudaMemcpy2DAsync(w.outs + (size_t)i * H, (size_t)S * H * 4, h, (size_t)H * 4, (size_t)H * 4, B, cudaMemcpyDeviceToDevice, st));
    }
    // grounding logits: ReLU(vis_embed)[cls] . g_pool^T + bias[cls] + att2 logits, masked (model.py:469-486)
    GVD_STAGE("teacher.ground", gvd_gather_class_rows(m->vis_relu, (const long long*)input_cls, w.emb, w.cls_idx, B, S, L1, V, 2048, m->NC, st));
    {
        GemmArgs g{};
        g.A = w.emb; g.lda = 2048; g.sAb = (long long)S * 2048;
        g.W = w.g_pool; g.ldw = 2048; g.sWb = (long long)R * 2048;
        g.C = w.G; g.ldc = R; g.sCb = (long long)S * R;
        g.M = S; g.N = R; g.K = 2048; g.nh = 1; g.alpha = 1.f;
        GVD_STAGE("teacher.ground", gvd_gemm_nt(g, B, st));
    }
    if (mode == 0) {
        GVD_STAGE("teacher.ground", gvd_grounding_finish(w.G, w.z_all, m->P("vis_classifiers_bias"), w.cls_idx, w.fm, R + 1, 1, B, S, R, st));
        // batched vocabulary head over all (clip, step) rows + LM loss (model.py:464-465, utils.py:122-136)
        GVD_STAGE("teacher.logit", gvd_linear(w.outs, H, m->P("logit.weight"), H, m->P("logit.bias"), w.logits_all, m->Vp, B * S, V, H, GVD_ACT_NONE, st));
        GVD_STAGE("teacher.loss", gvd_lm_nll(w.logits_all, m->Vp, (const long long*)seq, B, S, L1, V, w.part_sum, w.part_cnt, st));
        GVD_STAGE("teacher.reduce", gvd_finish_mean(w.part_sum, w.part_cnt, B * S, 1.f, losses_out + 0, st));
        GVD_STAGE("teacher.loss", gvd_att_nll(w.z_all, w.labels, (long long)B * S, R, w.part_sum, w.part_cnt, st));       // utils.py:139
        GVD_STAGE("teacher.reduce", gvd_finish_mean(w.part_sum, w.part_cnt, B * S, -1.f, losses_out + 1, st));
        GVD_STAGE("teacher.loss", gvd_att_nll(w.G, w.labels, (long long)B * S, R, w.part_sum, w.part_cnt, st));           // utils.py:142
        GVD_STAGE("teacher.reduce", gvd_finish_mean(w.part_sum, w.part_cnt, B * S, -1.f, losses_out + 2, st));
    } else {
        GVD_STAGE("teacher.ground", gvd_grounding_finish(w.G, w.z_all, m->P("vis_classifiers_bias"), w.cls_idx, pnt_mask, R + 1, 0, B, S, R, st));
        GVD_STAGE("teacher.argmax", gvd_frame_argmax(w.z_all, (long long*)att_idx_out, (long long)B * S, d.num_sampled_frm, d.num_prop_per_frm, st));
        GVD_STAGE("teacher.argmax", gvd_frame_argmax(w.G, (long long*)grd_idx_out, (long long)B * S, d.num_sampled_frm, d.num_prop_per_frm, st));
    }
    return 0;
}

// B1/B2: beam search for every clip at once (misc/model.py:700-742 + misc/CaptionModelBU.py:104-185, repaired semantics)
extern "C" GVD_API int gvd_beam_decode(gvd_model_t* m, int B, int T, int beam_size, void* workspace, size_t workspace_bytes,
                                       const uint8_t* pnt_mask, int64_t* seq_out, float* logprobs_out, int64_t* att2_idx_out, void* stream) {
    GVD_REQUIRE(beam_size >= 2, "beam_decode: beam_size must be >= 2 (use gvd_decode_greedy for 1)");
    WS w;
    GVD_TRY(check_ws(m, B, T, workspace, workspace_bytes, &w, beam_size));
    GVD_REQUIRE(pnt_mask && seq_out && logprobs_out && att2_idx_out, "beam_decode: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const gvd_dims_t& d = m->d;
    const int H = d.rnn_size, V = d.vocab_size, L = d.seq_length, R = m->R, K = beam_size, BK = B * K;
    const size_t BKH = (size_t)BK * H;
    {   // zero state, <bos> tokens, bookkeeping init (beam_seq 0, att2 indices -1, sums 0)
        const size_t n = BKH * sizeof(float);
        GVD_CHECK_CUDA(cudaMemsetAsync(w.h_att, 0, 2 * n, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.c_att, 0, n, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.h_lang, 0, 2 * n, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.c_lang, 0, n, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.bb.tokens, 0, (size_t)BK * 8, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.bb.seq, 0, (size_t)B * L * K * 4, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.bb.lp, 0, (size_t)B * L * K * 4, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.bb.att, 0xFF, (size_t)B * L * K * 4, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.bb.att_ind, 0xFF, (size_t)BK * 4, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.bb.sums, 0, (size_t)B * K * 4, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.bb.done_flag, 0, (size_t)B * 4, st));
        GVD_CHECK_CUDA(cudaMemsetAsync(w.ticket, 0, (size_t)BK * sizeof(int), st));
    }
    // first core step on <bos> (model.py:723-733): all K rows of a clip are identical
    GVD_TRY(core_step(m, w, BK, T, 0, w.bb.tokens, pnt_mask, pnt_mask, w.z_rows, R, st, K));
    GVD_STAGE("beam.argmax", gvd_row_argmax(w.z_rows, R, BK, R, w.bos_att, st));
    for (int t = 0; t < L; ++t) {
        const int par = (t + 1) & 1;                      // state parity written by the previous core step
        float* h_att = w.h_att + (size_t)par * BKH;
        float* h_lang = w.h_lang + (size_t)par * BKH;
        GVD_STAGE("decode.logit", gvd_linear(h_lang, H, m->P("logit.weight"), H, m->P("logit.bias"), w.logits, m->Vp, BK, V, H, GVD_ACT_NONE, st));
        GVD_STAGE("beam.topk", gvd_beam_topk(w.logits, m->Vp, BK, V, K, w.bb.topv, w.bb.topi, st));
        GVD_STAGE("beam.update", gvd_beam_update(w.bb, B, K, L, t, st));
        if (t == L - 1) break;                            // the reference runs one more (unused) core step
        float* bufs[4] = {h_att, w.c_att, h_lang, w.c_lang};
        for (float* buf : bufs) {                         // rearrange recurrent state to the surviving beams (CaptionModelBU.py:85-89)
            GVD_STAGE("beam.gather", gvd_beam_gather_rows(buf, w.gather_tmp, w.bb.parent, B, K, H, st));
            GVD_CHECK_CUDA(cudaMemcpyAsync(buf, w.gather_tmp, BKH * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
        GVD_TRY(core_step(m, w, BK, T, t + 1, w.bb.tokens, pnt_mask, pnt_mask, w.z_rows, R, st, K));
        GVD_STAGE("beam.argmax", gvd_row_argmax(w.z_rows, R, BK, R, w.bb.att_ind, st));
    }
    GVD_STAGE("beam.finish", gvd_beam_finish(w.bb, w.bos_att, B, K, L, (long long*)seq_out, logprobs_out, (long long*)att2_idx_out, st));
    return 0;
}

// Clip chunks of the host-buffer entry point.  The persistent GEMMs walk 128-row tiles on 148 CTAs, so a chunk costs whole waves: 9 / 18 / 27 clips
// (71 / 141 / 211 row tiles) fill their last wave to > 93 %, 12 clips (94 tiles) only to 64-80 %.  The pipeline starts with one attention
// sub-batch (`unit` clips: the first kernel waits for the first copy) and grows 1, 2, 3, 6, 9, 12, 12 ... units while the copy engine stays ahead
// (copy 0.16 ms per clip, compute 0.21 ms per clip); a short remainder joins the last chunk.  B = 100: 3, 6, 9, 18, 27, 37 clips — measured
// (tools/overlap_sweep.py, session 30) 27.55 ms end to end against 30.6 ms for uniform 12-clip chunks and 25.0 ms with the inputs resident.
// GVD_H2D_SCHED="3,6,9,..." (clips per chunk; a short list repeats its last entry) or GVD_H2D_CHUNK=n (uniform) override the rule.
static std::vector<int> h2d_schedule(int B, int unit) {
    std::vector<int> s;
    int left = B;
    auto push = [&](int n) { n = std::max(1, std::min(n, left)); s.push_back(n); left -= n; };
    if (const char* e = getenv("GVD_H2D_SCHED")) {
        int last = 0;
        for (const char* p = e; *p && left > 0;) {
            char* q = nullptr;
            const long v = strtol(p, &q, 10);
            if (q == p) break;
            if (v > 0) { last = (int)v; push(last); }
            p = (*q == ',') ? q + 1 : q;
        }
        while (left > 0) push(last > 0 ? last : left);
        return s;
    }
    if (const char* e = getenv("GVD_H2D_CHUNK")) {
        const int c = std::max(1, atoi(e));
        while (left > 0) push(c);
        return s;
    }
    const int grow[5] = {1, 2, 3, 6, 9};
    for (int i = 0; i < 5 && left > 0; ++i) push(left < (grow[i] + 2) * unit ? left : grow[i] * unit);
    while (left > 0) push(left < 16 * unit ? left : 12 * unit);
    return s;
}

extern "C" GVD_API int gvd_plan_h2d_chunks(int batch_clips, int unit, int* chunks_out, int cap) {
    if (!(batch_clips >= 1 && unit >= 1 && chunks_out && cap >= 1)) { gvd_set_error("plan_h2d_chunks: bad arguments"); return -1; }
    const std::vector<int> s = h2d_schedule(batch_clips, std::min(unit, batch_clips));
    if ((int)s.size() > cap) { gvd_set_error("plan_h2d_chunks: %d chunks do not fit the caller's array of %d", (int)s.size(), cap); return -1; }
    for (size_t i = 0; i < s.size(); ++i) chunks_out[i] = s[i];
    return (int)s.size();
}

extern "C" GVD_API int gvd_sample_greedy_host(gvd_model_t* m, int B, int T, const float* h_segs_feat, const float* h_ppls, const int64_t* h_num,
                                      const float* h_ppls_feat, const int64_t* h_sample_idx, const uint8_t* h_pnt_mask, void* workspace,
                                      size_t workspace_bytes, int64_t* h_seq_out, float* h_logprobs_out, float* h_att2_out,
                                      float* h_sim_mat_out, void* stream) {
    WS w;
    GVD_TRY(check_ws(m, B, T, workspace, workspace_bytes, &w));
    GVD_REQUIRE(h_segs_feat && h_ppls && h_num && h_ppls_feat && h_sample_idx && h_pnt_mask && h_seq_out, "sample_greedy_host: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const gvd_dims_t& d = m->d;
    const int R = m->R, L = d.seq_length, FC = d.fc_feat_size;
    const size_t BR = (size_t)B * R, BT = (size_t)B * T;
    // The fc6 region features are ~98 % of the input bytes (819 MB at B=100) and every region stage is per-clip independent,
    // so they cross PCIe in clip chunks on a second stream while the previous chunk runs P2-P6 on the compute stream.
    const std::vector<int> sched = h2d_schedule(B, w.clip_chunk);
    const int nchunks = (int)sched.size();
    if (!m->copy_stream) GVD_CHECK_CUDA(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
    while ((int)m->events.size() < nchunks + 3) {
        cudaEvent_t e;
        GVD_CHECK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        m->events.push_back(e);
    }
    cudaEvent_t ev_start = m->events[nchunks], ev_sim = m->events[nchunks + 1], ev_segs = m->events[nchunks + 2];
    // Frame stages (P1 + P7) on their own stream next to the region stages (see frame_fork).  Long clips (reference default T = 480: 590 MB of
    // frame features, a 17 ms GRU chain): the frame features cross PCIe after the first ~30 % of the region chunks — early enough for the
    // chain to end with the region stages, late enough for those to have work while the features travel; the chunks enqueued behind them run
    // with the SM reserve for about as long as the chain lasts.  Without the second stream they travel last and the frame stages run last.
    const bool overlap = frame_overlap_on();
    const bool big_segs = BT * (size_t)FC * 4 > ((size_t)64 << 20);
    int segs_after = 0;                                   // chunks copied before the frame features (big_segs only)
    if (big_segs) {
        segs_after = nchunks;
        if (overlap) {
            const int want = getenv("GVD_H2D_SEGS_AFTER") ? atoi(getenv("GVD_H2D_SEGS_AFTER")) : (3 * B + 9) / 10;      // clips
            int acc = 0;
            segs_after = 0;
            while (segs_after < nchunks && acc < want) acc += sched[segs_after++];
        }
    }
    const int res_sms = frame_reserve_sms(m);
    int res_left = (overlap && big_segs) ? frame_reserve_clips(m, w, B, T) : 0;     // clips still to run with the reserve once the chain has started
    const bool trace = getenv("GVD_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto ms_since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
    GVD_CHECK_CUDA(cudaEventRecord(ev_start, st));                       // the workspace may still be in use by earlier work on `st`
    GVD_CHECK_CUDA(cudaStreamWaitEvent(m->copy_stream, ev_start, 0));
    if (!big_segs) GVD_CHECK_CUDA(cudaMemcpyAsync(w.in_segs, h_segs_feat, BT * FC * 4, cudaMemcpyHostToDevice, st));
    GVD_CHECK_CUDA(cudaMemcpyAsync(w.in_ppls, h_ppls, BR * 7 * 4, cudaMemcpyHostToDevice, st));
    GVD_CHECK_CUDA(cudaMemcpyAsync(w.in_num, h_num, (size_t)B * 7 * 8, cudaMemcpyHostToDevice, st));
    GVD_CHECK_CUDA(cudaMemcpyAsync(w.in_sidx, h_sample_idx, (size_t)B * 2 * 8, cudaMemcpyHostToDevice, st));
    GVD_CHECK_CUDA(cudaMemcpyAsync(w.in_mask, h_pnt_mask, (size_t)B * (R + 1), cudaMemcpyHostToDevice, st));
    cudaStream_t fst = st;
    if (overlap) { GVD_TRY(frame_fork(m, st)); fst = m->frame_stream; }          // (forked behind the small copies: the frame stages read num / sample_idx)
    // the big chunk copies are enqueued AFTER the small ones: the H2D copy engine is one FIFO across streams, and the first
    // kernels on `st` need the small tensors
    auto copy_segs = [&]() -> int {
        GVD_CHECK_CUDA(cudaMemcpyAsync(w.in_segs, h_segs_feat, BT * FC * 4, cudaMemcpyHostToDevice, m->copy_stream));
        GVD_CHECK_CUDA(cudaEventRecord(ev_segs, m->copy_stream));
        return 0;
    };
    {
        size_t c0 = 0;
        for (int c = 0; c < nchunks; ++c) {
            if (big_segs && c == segs_after) GVD_TRY(copy_segs());
            const size_t cb = (size_t)sched[c];
            GVD_CHECK_CUDA(cudaMemcpyAsync(w.in_feat + c0 * R * d.att_feat_size, h_ppls_feat + c0 * R * d.att_feat_size, cb * R * d.att_feat_size * 4,
                                           cudaMemcpyHostToDevice, m->copy_stream));
            GVD_CHECK_CUDA(cudaEventRecord(m->events[c], m->copy_stream));
            c0 += cb;
        }
        if (big_segs && segs_after >= nchunks) GVD_TRY(copy_segs());
    }
    if (trace) fprintf(stderr, "[gvd] %.2f ms: copies enqueued (%d chunks, frame features after chunk %d)\n", ms_since(), nchunks, big_segs ? segs_after : 0);
    int rc = 0;
    bool frame_done = false;
    auto run_frame = [&]() -> int {
        frame_done = true;
        if (big_segs) GVD_CHECK_CUDA(cudaStreamWaitEvent(fst, ev_segs, 0));
        return frame_stages(m, w, B, T, w.in_segs, w.in_num, w.in_sidx, fst);
    };
    if (!big_segs) rc = run_frame();
    {
        int c0 = 0;
        for (int c = 0; c < nchunks && rc == 0; ++c) {
            // on one stream the frame stages go last (they would hold up the region chunks behind the frame-feature copy)
            if (big_segs && overlap && c == segs_after && !frame_done) { rc = run_frame(); if (rc) break; }
            const int cb = sched[c];
            GVD_CHECK_CUDA(cudaStreamWaitEvent(st, m->events[c], 0));
            const bool reserve = frame_done && overlap && big_segs && res_left > 0;
            SmReserveScope rs(reserve ? res_sms : 0);
            if (reserve) res_left -= cb;
            rc = region_prologue(m, w, c0, cb, w.in_ppls + (size_t)c0 * R * 7, w.in_feat + (size_t)c0 * R * d.att_feat_size,
                                 w.in_mask + (size_t)c0 * (R + 1), h_sim_mat_out ? w.out_sim + (size_t)c0 * m->NC * R : nullptr, st);
            c0 += cb;
        }
    }
    if (rc == 0 && !frame_done) rc = run_frame();
    if (overlap) { const int jr = frame_join(m, st); if (rc == 0) rc = jr; }
    if (rc != 0) { cudaStreamSynchronize(m->copy_stream); return rc; }            // (the copies read caller memory: never return with them in flight)
    if (trace) fprintf(stderr, "[gvd] %.2f ms: prologue enqueued\n", ms_since());
    if (h_sim_mat_out) {   // the similarity matrix is final here: its D2H overlaps the 20-step decode loop
        GVD_CHECK_CUDA(cudaEventRecord(ev_sim, st));
        GVD_CHECK_CUDA(cudaStreamWaitEvent(m->copy_stream, ev_sim, 0));
        GVD_CHECK_CUDA(cudaMemcpyAsync(h_sim_mat_out, w.out_sim, (size_t)B * m->NC * R * 4, cudaMemcpyDeviceToHost, m->copy_stream));
    }
    GVD_TRY(gvd_decode_greedy(m, B, T, workspace, workspace_bytes, w.in_mask, (int64_t*)w.out_seq, w.out_logp, w.out_att2, stream));
    GVD_CHECK_CUDA(cudaMemcpyAsync(h_seq_out, w.out_seq, (size_t)B * L * 8, cudaMemcpyDeviceToHost, st));
    if (h_logprobs_out) GVD_CHECK_CUDA(cudaMemcpyAsync(h_logprobs_out, w.out_logp, (size_t)B * L * 4, cudaMemcpyDeviceToHost, st));
    if (h_att2_out) GVD_CHECK_CUDA(cudaMemcpyAsync(h_att2_out, w.out_att2, (size_t)B * L * R * 4, cudaMemcpyDeviceToHost, st));
    if (trace) fprintf(stderr, "[gvd] %.2f ms: everything enqueued\n", ms_since());
    GVD_CHECK_CUDA(cudaStreamSynchronize(st));
    if (trace) fprintf(stderr, "[gvd] %.2f ms: compute stream drained\n", ms_since());
    GVD_CHECK_CUDA(cudaStreamSynchronize(m->copy_stream));
    if (trace) fprintf(stderr, "[gvd] %.2f ms: copy stream drained\n", ms_since());
    return 0;
}

// Post-decode grounding extraction (main.py:364-370, SURVEY 8(f) rank 2): for every generated word and every sampled frame the
// proposal with the largest region-attention logit, and its box row.  att2 [B, L, F*P] (the second output of 'sample'),
// ppls [B, F*P, 7]; idx_out [B, L, F] int64, boxes_out [B, L, F, 7] (may be null).  Ties -> lowest index (torch.max on CPU).
extern "C" GVD_API int gvd_grounding_extract(const float* att2, const float* ppls, int B, int L, int num_frames, int num_prop, int64_t* idx_out,
                                             float* boxes_out, void* stream) {
    GVD_REQUIRE(att2 && ppls && idx_out && B > 0 && L > 0 && num_frames > 0 && num_prop > 0, "grounding_extract: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    GVD_TRY(gvd_frame_argmax(att2, (long long*)idx_out, (long long)B * L, num_frames, num_prop, st));
    if (boxes_out) GVD_TRY(gvd_grounding_gather(ppls, (const long long*)idx_out, boxes_out, B, L, num_frames, num_prop, 7, st));
    return 0;
}

// Grounding-evaluator hit test (tools/anet_entities/scripts/eval_grd_anet_entities.py:95-102, SURVEY 8(f) rank 3), batched over
// words: pred [N,F,5] (x1,y1,x2,y2,frame), ref [N,K,5] with the first nref[n] rows valid -> max IoU [N] and hit [N] = max > thresh.
extern "C" GVD_API int gvd_grounding_eval(const float* pred, const float* ref, const int* nref, int N, int F, int K, float iou_thresh,
                                          float* max_iou_out, unsigned char* hit_out, void* stream) {
    GVD_REQUIRE(pred && ref && nref && max_iou_out && hit_out && N > 0 && F > 0 && K > 0, "grounding_eval: bad arguments");
    return gvd_grounding_eval_hits(pred, ref, nref, max_iou_out, hit_out, N, F, K, iou_thresh, (cudaStream_t)stream);
}

// K-split plan of the operand-swapped skinny products (host logic only, no device access): number of splits, 0 = shape not supported
extern "C" GVD_API int gvd_plan_skinny_splits(int weight_rows, int k_total, int batch_rows) { return gvd_skinny_splits(weight_rows, k_total, batch_rows); }

// ------------------------------------------------------------------------------------ single ops
extern "C" GVD_API int gvd_op_linear(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, float* C, int64_t ldc, int M,
                             int N, int K, int act, void* stream) {
    GVD_REQUIRE(A && W && C, "op_linear: null argument");
    return gvd_linear(A, lda, W, ldw, bias, C, ldc, M, N, K, act, (cudaStream_t)stream);
}
extern "C" GVD_API int gvd_op_linear_tc(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, float* C, int64_t ldc,
                                        int M, int N, int K, int act, void* stream) {
    GVD_REQUIRE(A && W && C, "op_linear_tc: null argument");
    GvdF16Scope f16;                               // test hook of a forward product: backend bit 4 selects the fp16x3 variant
    GemmArgs g{};
    g.A = A; g.lda = lda; g.W = W; g.ldw = ldw; g.C = C; g.ldc = ldc; g.bias = bias;
    g.M = M; g.N = N; g.K = K; g.nh = 1; g.act = act; g.alpha = 1.f;
    return gvd_gemm_nt_tc(g, 1, (cudaStream_t)stream);
}
// The conversion-free prologue GEMM (f16ss_persistent_kernel) on its own: both operands are packed into fp16x3 images here (scratch from the
// stream-ordered allocator), optionally with the fp16x3 image of the output (img_out [M, rup32(N)] words) next to / instead of C.  Test hook.
extern "C" GVD_API int gvd_op_linear_f16ss(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, float* C, int64_t ldc,
                                           float* img_out, int M, int N, int K, int act, void* stream) {
    GVD_REQUIRE(A && W && (C || img_out) && M > 0 && N > 0 && K > 0, "op_linear_f16ss: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const long long Kp = (K + 31) / 32 * 32, Np = (N + 31) / 32 * 32;
    float *Ai = nullptr, *Wi = nullptr;
    GVD_CHECK_CUDA(cudaMallocAsync((void**)&Ai, (size_t)M * Kp * 4, st));
    GVD_CHECK_CUDA(cudaMallocAsync((void**)&Wi, (size_t)N * Kp * 4, st));
    int rc = gvd_pack_f16x3(A, lda, M, K, Ai, Kp, st, GVD_F16_SA);
    if (!rc) rc = gvd_pack_f16x3(W, ldw, N, K, Wi, Kp, st, GVD_F16_SW);
    if (!rc) rc = gvd_gemm_f16ss(Ai, Kp, Wi, Kp, bias, nullptr, nullptr, act, C, ldc, M, N, K, st, img_out, img_out ? Np : 0);
    cudaFreeAsync(Ai, st);
    cudaFreeAsync(Wi, st);
    return rc;
}
// One LSTMCell step from up to two dense input segments [x0 | x1] (weights w0 [4H,K0], w1 [4H,K1]); backend 0 = CUDA cores, 1 = tcgen05
extern "C" GVD_API int gvd_op_lstm_step(int B, int H, const float* x0, int K0, const float* w0, int64_t ldw0, const float* x1, int K1,
                                        const float* w1, int64_t ldw1, const float* bias1, const float* bias2, const float* c_prev,
                                        float* h_out, float* c_out, int backend, void* stream) {
    GVD_REQUIRE(x0 && w0 && c_prev && h_out && c_out, "op_lstm_step: null argument");
    GvdF16Scope f16;
    LstmArgs a{};
    a.nseg = x1 ? 2 : 1;
    a.seg[0] = LstmSeg{x0, K0, nullptr, 0, w0, ldw0, K0};
    if (x1) a.seg[1] = LstmSeg{x1, K1, nullptr, 0, w1, ldw1, K1};
    a.bias1 = bias1; a.bias2 = bias2; a.c_prev = c_prev; a.h_out = h_out; a.c_out = c_out; a.B = B; a.H = H;
    return backend ? gvd_lstm_step_tc(a, (cudaStream_t)stream) : gvd_lstm_step(a, (cudaStream_t)stream);
}
// Batched short-K product C[b,h] = A[b,:,h*hs:(h+1)*hs] . W[b,:,h*hs:(h+1)*hs]^T through the A-stationary kernel (the attention-score shape)
extern "C" GVD_API int gvd_op_scores_tc(const float* A, const float* W, float* C, int nb, int nh, int M, int N, int hs, int64_t ld, void* stream) {
    GVD_REQUIRE(A && W && C, "op_scores_tc: null argument");
    GemmArgs g{};
    g.A = A; g.lda = ld; g.sAb = (long long)M * ld; g.sAh = hs;
    g.W = W; g.ldw = ld; g.sWb = (long long)N * ld; g.sWh = hs;
    g.C = C; g.ldc = N; g.sCb = (long long)nh * M * N; g.sCh = (long long)M * N;
    g.M = M; g.N = N; g.K = hs; g.nh = nh; g.alpha = 1.f;
    return gvd_gemm_nt_astat(g, nb * nh, (cudaStream_t)stream);
}
// Self-attention core of one encoder layer on a packed projection buffer qkv [nb, R, 3*HP] (Q | K | V, heads of width hs at
// column h*hs):  out[nb, R, HP] = concat_h softmax(Q_h K_h^T * scale) V_h through the fused tcgen05 pair.  Test hook: the
// scratch buffers are allocated here.  E [nb,nh,R,R] (numerators) and F [nb,nh,ceil(R/32),R] (group factors) are caller
// buffers; stages: bit 0 = scores (writes E, F), bit 1 = P.V (reads E, F, writes out).
extern "C" GVD_API int gvd_op_self_attention_tc(const float* qkv, float* out, int nb, int nh, int R, int hs, int HP, float scale, float* E,
                                                float* F, int stages, void* stream) {
    GVD_REQUIRE(qkv && out && E && F && nb > 0 && nh > 0 && R > 0 && R % 4 == 0 && HP % 4 == 0 && nh * hs <= HP, "op_self_attention_tc: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t BR = (size_t)nb * R;
    float *khi = nullptr, *klo = nullptr, *vh = nullptr, *vl = nullptr;
    const bool att16 = (gvd_backend() & 256) != 0;          // fp16x3 images instead of tf32 planes (same switch as the prologue)
    const int KH = (hs + 31) / 32 * 32, Rp = (R + 31) / 32 * 32;
    auto body16 = [&]() -> int {
        GVD_CHECK_CUDA(cudaMalloc(&khi, BR * nh * KH * 4)); GVD_CHECK_CUDA(cudaMalloc(&vh, (size_t)nb * HP * Rp * 4));
        if (stages & 1) {
            GVD_TRY(gvd_pack_heads_f16x3(qkv + HP, 3 * HP, (long long)BR, nh, hs, hs, KH, GVD_ATT_SK_HOST, khi, st));
            GemmArgs g{};
            g.A = qkv; g.lda = 3 * HP; g.sAb = (long long)R * 3 * HP; g.sAh = hs;
            g.W = khi; g.ldw = (long long)nh * KH; g.sWb = (long long)R * nh * KH; g.sWh = KH;
            g.C = E; g.ldc = R; g.sCb = (long long)nh * R * R; g.sCh = (long long)R * R;
            g.M = R; g.N = R; g.K = hs; g.nh = nh; g.alpha = 1.f;
            GVD_TRY(gvd_attn_scores_tc(g, nullptr, F, scale, nb * nh, st, 1));
        }
        if (stages & 2) {
            GVD_TRY(gvd_transpose_pack_f16x3(qkv + 2 * HP, vh, nb, R, HP, 3 * HP, Rp, GVD_ATT_SV_HOST, st));
            GemmArgs v{};
            v.A = E; v.lda = R; v.sAb = (long long)nh * R * R; v.sAh = (long long)R * R;
            v.W = vh; v.ldw = Rp; v.sWb = (long long)HP * Rp; v.sWh = (long long)hs * Rp;
            v.C = out; v.ldc = HP; v.sCb = (long long)R * HP; v.sCh = hs;
            v.M = R; v.N = hs; v.K = R; v.nh = nh; v.alpha = 1.f;
            GVD_TRY(gvd_attn_pv_tc(v, nullptr, F, nb * nh, st, 1));
        }
        GVD_CHECK_CUDA(cudaStreamSynchronize(st));
        return 0;
    };
    auto body = [&]() -> int {
        GVD_CHECK_CUDA(cudaMalloc(&khi, BR * HP * 4)); GVD_CHECK_CUDA(cudaMalloc(&klo, BR * HP * 4));
        GVD_CHECK_CUDA(cudaMalloc(&vh, BR * HP * 4)); GVD_CHECK_CUDA(cudaMalloc(&vl, BR * HP * 4));
        if (stages & 1) {
            GVD_TRY(gvd_split_hilo(qkv + HP, 3 * HP, khi, klo, HP, (long long)BR, HP, st));
            GemmArgs g{};
            g.A = qkv; g.lda = 3 * HP; g.sAb = (long long)R * 3 * HP; g.sAh = hs;
            g.W = khi; g.ldw = HP; g.sWb = (long long)R * HP; g.sWh = hs;
            g.C = E; g.ldc = R; g.sCb = (long long)nh * R * R; g.sCh = (long long)R * R;
            g.M = R; g.N = R; g.K = hs; g.nh = nh; g.alpha = 1.f;
            GVD_TRY(gvd_attn_scores_tc(g, klo, F, scale, nb * nh, st));
        }
        if (stages & 2) {
            GVD_TRY(gvd_transpose_split(qkv + 2 * HP, vh, vl, nb, R, HP, 3 * HP, st));
            GemmArgs v{};
            v.A = E; v.lda = R; v.sAb = (long long)nh * R * R; v.sAh = (long long)R * R;
            v.W = vh; v.ldw = R; v.sWb = (long long)HP * R; v.sWh = (long long)hs * R;
            v.C = out; v.ldc = HP; v.sCb = (long long)R * HP; v.sCh = hs;
            v.M = R; v.N = hs; v.K = R; v.nh = nh; v.alpha = 1.f;
            GVD_TRY(gvd_attn_pv_tc(v, vl, F, nb * nh, st));
        }
        GVD_CHECK_CUDA(cudaStreamSynchronize(st));
        return 0;
    };
    const int rc = att16 ? body16() : body();
    cudaFree(khi); cudaFree(klo); cudaFree(vh); cudaFree(vl);
    return rc;
}
extern "C" GVD_API int gvd_op_tanh(const float* x, float* y, int n, void* stream) { return gvd_tanh_test(x, y, n, (cudaStream_t)stream); }
