// pyfastllama.so: the llama_* C ABI of fastLLaMa's Python interface (interfaces/c/fastllama.h upstream) over libggml_b200.
//
// Model loading (ggml / ggmf / ggjt files), LoRA adapters, the SentencePiece-style tokenizer, the LLaMA eval graph, the session
// logic of ingest / generate / perplexity / state files, and sampling.  Everything numeric runs below ggml_graph_compute on the B200;
// what is computed here on the host (sampling, perplexity's soft-max) uses fastLLaMa's order of operations, so tokens, logits,
// perplexities and state files match fastLLaMa's own library.  Two deliberate differences: with stop words, every held-back token
// is streamed when generate() ends (fastLLaMa streams one of them), and greedy sampling with all logits kept takes the argmax of
// the last row (fastLLaMa's index runs over every row and can leave the vocabulary).
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <deque>
#include <fcntl.h>
#include <memory>
#include <numeric>
#include <queue>
#include <random>
#include <sstream>
#include <string>
#include <string_view>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "fl_ggml.h"

// ---- C ABI types (layouts of fastLLaMa's interfaces/c/fastllama.h) ---------------------------------------------------------
extern "C" {
typedef void (*llama_log_fn)(const char *func, int func_len, const char *msg, int msg_len);
typedef void (*llama_reset_fn)(void);
typedef void (*llama_progress_fn)(uint8_t tag, size_t done, size_t total);
typedef void (*llama_stream_fn)(const char *text, int len);

struct llama_logger { llama_log_fn log, log_err, log_warn; llama_reset_fn reset; llama_progress_fn progress; };
struct llama_array_view_f { const float *data; size_t size; };
struct llama_model_context_args {
    bool embedding_eval_enabled, should_get_all_logits, use_mmap, use_mlock, load_parallel;
    int seed, n_keep, n_ctx, n_threads, n_batch;
    uint32_t n_load_parallel_blocks;
    size_t last_n_tokens, allocate_extra_mem;
    struct llama_logger logger;
};
}

namespace {

using token_id = int32_t;
constexpr token_id BOS = 1, EOS = 2;
constexpr uint8_t PROGRESS_INGEST = 4;
constexpr size_t MiB = size_t(1) << 20;

struct Log {
    llama_logger cb{};
    void emit(llama_log_fn f, const char *func, const char *fmt, va_list ap) const {
        if (!f) return;
        char buf[1024];
        const int n = vsnprintf(buf, sizeof buf, fmt, ap);
        f(func, (int)strlen(func), buf, std::min(n, (int)sizeof buf - 1));
    }
    void info(const char *func, const char *fmt, ...) const { va_list ap; va_start(ap, fmt); emit(cb.log, func, fmt, ap); va_end(ap); }
    void err(const char *func, const char *fmt, ...) const { va_list ap; va_start(ap, fmt); emit(cb.log_err, func, fmt, ap); va_end(ap); }
    void reset() const { if (cb.reset) cb.reset(); }
    void progress(uint8_t tag, size_t done, size_t total) const { if (cb.progress) cb.progress(tag, done, total); }
};

void default_info(const char *f, int fl, const char *m, int ml) { printf("[Info]: Func('%.*s') %.*s", fl, f, ml, m); fflush(stdout); }
void default_warn(const char *f, int fl, const char *m, int ml) { printf("[Warn]: Func('%.*s') %.*s", fl, f, ml, m); fflush(stdout); }
void default_err(const char *f, int fl, const char *m, int ml) { fprintf(stderr, "[Error]: Func('%.*s') %.*s", fl, f, ml, m); fflush(stderr); }
void default_reset() {}
void default_progress(uint8_t, size_t, size_t) {}

// ---- vocabulary and tokenizer ------------------------------------------------------------------------------------------------
struct Vocab {
    std::vector<std::string> text;
    std::vector<float> score;
    std::unordered_map<std::string, token_id> id_of;
};

size_t utf8_len(char c) {
    static const size_t len_by_high_nibble[16] = {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 3, 4};
    return len_by_high_nibble[(uint8_t)c >> 4];
}

// Greedy pair merging: start from UTF-8 characters and repeatedly join the adjacent pair whose concatenation is the
// highest-scoring vocabulary entry (the leftmost pair on a tie).  Pieces that are not in the vocabulary fall back to one token
// per byte (id = byte + 3).
std::vector<token_id> tokenize(const Vocab &v, std::string_view text, bool bos) {
    std::vector<token_id> out;
    if (text.empty()) return out;
    if (bos) out.push_back(BOS);
    struct Piece { size_t begin, len; int prev, next; };
    std::vector<Piece> pieces;
    for (size_t off = 0; off < text.size();) {
        const size_t n = std::min(text.size() - off, utf8_len(text[off]));
        const int i = (int)pieces.size();
        off += n;
        pieces.push_back({off - n, n, i - 1, off == text.size() ? -1 : i + 1});
    }
    struct Pair { int left, right; float score; size_t len; };
    auto lower = [](const Pair &a, const Pair &b) { return a.score < b.score || (a.score == b.score && a.left > b.left); };
    std::priority_queue<Pair, std::vector<Pair>, decltype(lower)> queue(lower);
    auto propose = [&](int l, int r) {
        if (l < 0 || r < 0) return;
        const std::string joined(text.substr(pieces[l].begin, pieces[l].len + pieces[r].len));
        auto it = v.id_of.find(joined);
        if (it == v.id_of.end() || (size_t)it->second >= v.text.size()) return;
        queue.push({l, r, v.score[it->second], joined.size()});
    };
    for (size_t i = 1; i < pieces.size(); ++i) propose((int)i - 1, (int)i);
    while (!queue.empty()) {
        const Pair p = queue.top();
        queue.pop();
        Piece &l = pieces[p.left], &r = pieces[p.right];
        if (l.len == 0 || r.len == 0 || l.len + r.len != p.len) continue;      // stale: one side was merged since
        l.len += r.len;
        l.next = r.next;
        if (r.next >= 0) pieces[r.next].prev = p.left;
        r.len = 0;
        propose(l.prev, p.left);
        propose(p.left, l.next);
    }
    for (int i = 0; i != -1; i = pieces[i].next) {
        const std::string piece(text.substr(pieces[i].begin, pieces[i].len));
        auto it = v.id_of.find(piece);
        if (it != v.id_of.end()) {
            out.push_back(it->second);
        } else {
            for (unsigned char c : piece) out.push_back((token_id)c + 3);
        }
    }
    return out;
}

// ---- model -------------------------------------------------------------------------------------------------------------------
struct HParams { int32_t n_vocab, n_embd, n_mult, n_head, n_layer, n_rot, ftype; };

struct Layer { ggml_tensor *attention_norm, *wq, *wk, *wv, *wo, *ffn_norm, *w1, *w2, *w3; };

struct ContextGuard {
    ggml_context *ctx = nullptr;
    ~ContextGuard() { if (ctx) ggml_free(ctx); }
};

struct Mapping {
    void *addr = MAP_FAILED;
    size_t size = 0;
    ~Mapping() { if (addr != MAP_FAILED) munmap(addr, size); }
};

struct Model {
    HParams hp{};
    int n_ctx = 512, n_batch = 16, n_threads = 1;
    bool use_mmap = false, all_logits = false, embeddings_enabled = false;
    size_t extra_mem = 0;
    Vocab vocab;
    Mapping mapping;
    std::unique_ptr<uint8_t[]> weight_buf, kv_buf, compute_buf;
    size_t compute_size = 0;
    ContextGuard weights, kv;            // declared after the buffers: the contexts are freed first
    ggml_tensor *tok_embeddings = nullptr, *norm = nullptr, *output = nullptr, *k = nullptr, *v = nullptr;
    std::vector<Layer> layers;
    std::unordered_map<std::string, ggml_tensor *> by_name;
    std::vector<float> embeddings;

    bool load(const char *path, const Log &log);
    bool eval(int n_past, const token_id *tokens, int n, std::vector<float> &logits, size_t &mem_per_token);
};

struct FileReader {
    FILE *f = nullptr;
    explicit FileReader(const char *path) : f(fopen(path, "rb")) {}
    ~FileReader() { if (f) fclose(f); }
    bool read(void *dst, size_t n) { return fread(dst, 1, n, f) == n; }
    template <class T> bool read(T &x) { return read(&x, sizeof x); }
};

struct TensorRecord { std::string name; int32_t type; std::vector<int64_t> ne; size_t offset, size; };

// File containers.  Model files: 'ggml' (no version field, no token scores), 'ggmf' v1 (scores), 'ggjt' v1 (scores, tensor data
// aligned to 32 bytes, so it can be mapped).  LoRA adapters: 'ggla' v1 (aligned like ggjt).
enum Container : uint32_t { GGML = 0x67676d6c, GGMF = 0x67676d66, GGJT = 0x67676a74, GGLA = 0x67676c61 };

bool read_container(FileReader &in, const char *path, const Log &log, uint32_t &magic) {
    uint32_t version = 1;
    if (!in.read(magic) || (magic != GGML && !in.read(version))) { log.err("load", "'%s' is too short\n", path); return false; }
    if ((magic != GGML && magic != GGMF && magic != GGJT && magic != GGLA) || version != 1) {
        log.err("load", "'%s' is not a model or adapter file this library reads (magic %08x, version %u)\n", path, magic, version);
        return false;
    }
    return true;
}

// The tensor directory after the header: {i32 n_dims, i32 name_len, i32 type, i32 ne[n_dims], name, [pad to 32], data}, in file order.
// Only the types libggml_b200 computes with are accepted (f32 and the q4_0 / q4_1 blocks).
bool read_tensor_dir(FileReader &in, const char *path, bool aligned, const Log &log, std::vector<TensorRecord> &out) {
    struct stat st;
    if (stat(path, &st) != 0) return false;
    for (;;) {
        int32_t hdr[3];
        if (fread(hdr, sizeof hdr, 1, in.f) != 1) break;
        const int32_t n_dims = hdr[0], name_len = hdr[1], type = hdr[2];
        if (n_dims < 1 || n_dims > 2 || name_len <= 0 || name_len > 512 || (type != GGML_TYPE_F32 && type != GGML_TYPE_Q4_0 && type != GGML_TYPE_Q4_1)) {
            log.err("load", "unsupported tensor record (dims %d, type %d) in '%s': this library computes with f32, q4_0 and q4_1 tensors\n", n_dims, type, path);
            return false;
        }
        TensorRecord r;
        r.type = type;
        int32_t ne[2] = {1, 1};
        std::string name(name_len, '\0');
        if (!in.read(ne, sizeof(int32_t) * n_dims) || !in.read(name.data(), name_len)) { log.err("load", "truncated tensor record in '%s'\n", path); return false; }
        r.name = name;
        r.ne.assign(ne, ne + n_dims);
        r.offset = (size_t)ftell(in.f);
        if (aligned) r.offset = (r.offset + 31) & ~size_t(31);
        const int64_t n_el = (int64_t)ne[0] * ne[1];
        if (ne[0] <= 0 || ne[1] <= 0 || n_el % ggml_blck_size((ggml_type)type)) { log.err("load", "tensor '%s' has a bad shape\n", name.c_str()); return false; }
        r.size = (size_t)(n_el / ggml_blck_size((ggml_type)type)) * ggml_type_size((ggml_type)type);
        if (r.offset + r.size > (size_t)st.st_size || fseek(in.f, (long)(r.offset + r.size), SEEK_SET) != 0) {
            log.err("load", "tensor '%s' runs past the end of '%s'\n", name.c_str(), path);
            return false;
        }
        out.push_back(r);
    }
    return true;
}

bool Model::load(const char *path, const Log &log) {
    FileReader in(path);
    if (!in.f) { log.err("Model", "failed to open '%s'\n", path); return false; }
    uint32_t magic = 0;
    if (!read_container(in, path, log, magic)) return false;
    if (magic == GGLA) { log.err("Model", "'%s' is a LoRA adapter, not a model\n", path); return false; }
    if (!in.read(hp) || hp.n_vocab <= 0 || hp.n_embd <= 0 || hp.n_head <= 0 || hp.n_layer <= 0 || hp.n_mult <= 0 || hp.n_embd % hp.n_head) {
        log.err("Model", "bad hyper-parameters in '%s'\n", path);
        return false;
    }
    vocab.text.resize(hp.n_vocab);
    vocab.score.assign(hp.n_vocab, 0.0f);
    for (int i = 0; i < hp.n_vocab; ++i) {
        uint32_t len = 0;
        if (!in.read(len) || len > (1u << 20)) { log.err("Model", "truncated vocabulary\n"); return false; }
        std::string s(len, '\0');
        if (!in.read(s.data(), len) || (magic != GGML && !in.read(vocab.score[i]))) { log.err("Model", "truncated vocabulary\n"); return false; }
        vocab.text[i] = s;
        vocab.id_of[s] = i;
    }
    std::vector<TensorRecord> dir;
    if (!read_tensor_dir(in, path, magic == GGJT, log, dir)) return false;
    std::unordered_map<std::string, TensorRecord> recs;
    for (auto &r : dir) recs[r.name] = r;
    if (use_mmap && magic != GGJT) {
        log.info("Model", "'%s' is not a ggjt file (its tensors are not aligned): reading it instead of mapping it\n", path);
        use_mmap = false;
    }
    struct stat st;
    if (stat(path, &st) != 0) return false;

    const int64_t n_embd = hp.n_embd, n_vocab = hp.n_vocab;
    const int64_t n_ff = ((2 * (4 * n_embd) / 3 + hp.n_mult - 1) / hp.n_mult) * hp.n_mult;

    // one weight arena: tensor headers only with mmap (data stays in the mapping), headers + data without
    size_t ctx_size = recs.size() * 1024 + MiB;
    if (!use_mmap) for (auto &kvp : recs) ctx_size += kvp.second.size;
    if (use_mmap) {
        const int fd = open(path, O_RDONLY);
        if (fd < 0) return false;
        mapping.size = (size_t)st.st_size;
        mapping.addr = mmap(nullptr, mapping.size, PROT_READ, MAP_SHARED, fd, 0);
        close(fd);
        if (mapping.addr == MAP_FAILED) { log.err("Model", "mmap of '%s' failed\n", path); return false; }
    }
    weight_buf.reset(new uint8_t[ctx_size]);
    weights.ctx = ggml_init({ctx_size, weight_buf.get(), use_mmap});
    if (!weights.ctx) { log.err("Model", "failed to initialise the weight context\n"); return false; }

    size_t used = 0;
    auto get = [&](const std::string &name, std::vector<int64_t> ne) -> ggml_tensor * {
        auto it = recs.find(name);
        if (it == recs.end()) { log.err("Model", "tensor '%s' is missing from the model file\n", name.c_str()); return nullptr; }
        const TensorRecord &r = it->second;
        if (r.ne != ne) { log.err("Model", "tensor '%s' has the wrong shape\n", name.c_str()); return nullptr; }
        ggml_tensor *t = ne.size() == 1 ? ggml_new_tensor_1d(weights.ctx, (ggml_type)r.type, ne[0])
                                        : ggml_new_tensor_2d(weights.ctx, (ggml_type)r.type, ne[0], ne[1]);
        if (use_mmap) {
            t->data = (uint8_t *)mapping.addr + r.offset;
        } else if (fseek(in.f, (long)r.offset, SEEK_SET) != 0 || !in.read(t->data, r.size)) {
            log.err("Model", "failed to read tensor '%s'\n", name.c_str());
            return nullptr;
        }
        ++used;
        by_name[name] = t;
        return t;
    };
    char name[128];
    if (!(tok_embeddings = get("tok_embeddings.weight", {n_embd, n_vocab})) || !(norm = get("norm.weight", {n_embd})) ||
        !(output = get("output.weight", {n_embd, n_vocab})))
        return false;
    layers.resize(hp.n_layer);
    for (int i = 0; i < hp.n_layer; ++i) {
        Layer &L = layers[i];
        auto nm = [&](const char *s) { snprintf(name, sizeof name, "layers.%d.%s.weight", i, s); return std::string(name); };
        if (!(L.attention_norm = get(nm("attention_norm"), {n_embd})) || !(L.wq = get(nm("attention.wq"), {n_embd, n_embd})) ||
            !(L.wk = get(nm("attention.wk"), {n_embd, n_embd})) || !(L.wv = get(nm("attention.wv"), {n_embd, n_embd})) ||
            !(L.wo = get(nm("attention.wo"), {n_embd, n_embd})) || !(L.ffn_norm = get(nm("ffn_norm"), {n_embd})) ||
            !(L.w1 = get(nm("feed_forward.w1"), {n_embd, n_ff})) || !(L.w2 = get(nm("feed_forward.w2"), {n_ff, n_embd})) ||
            !(L.w3 = get(nm("feed_forward.w3"), {n_embd, n_ff})))
            return false;
    }
    if (used != recs.size()) { log.err("Model", "the model file has %zu tensors, %zu were expected\n", recs.size(), used); return false; }

    // KV cache: f32 K and V for every layer and position
    const size_t n_el = (size_t)n_embd * hp.n_layer * n_ctx;
    const size_t kv_size = 2 * n_el * sizeof(float) + 2 * MiB;
    kv_buf.reset(new uint8_t[kv_size]());
    kv.ctx = ggml_init({kv_size, kv_buf.get(), false});
    if (!kv.ctx) { log.err("Model", "failed to allocate the KV cache\n"); return false; }
    k = ggml_new_tensor_1d(kv.ctx, GGML_TYPE_F32, (int64_t)n_el);
    v = ggml_new_tensor_1d(kv.ctx, GGML_TYPE_F32, (int64_t)n_el);

    // compute arena of one eval, sized like fastLLaMa's per-model table plus 20 MiB per token of the batch
    const size_t eval_mib = hp.n_layer >= 80 ? 1536 : hp.n_layer >= 60 ? 1280 : hp.n_layer >= 40 ? 1024 : 768;
    compute_size = eval_mib * MiB + (size_t)n_batch * 20 * MiB + extra_mem;
    compute_buf.reset(new uint8_t[compute_size]());
    log.info("Model", "n_vocab = %d, n_embd = %d, n_head = %d, n_layer = %d, n_ff = %lld, n_ctx = %d\n", hp.n_vocab, hp.n_embd, hp.n_head,
             hp.n_layer, (long long)n_ff, n_ctx);
    return true;
}

bool Model::eval(int n_past, const token_id *tokens, int n, std::vector<float> &logits, size_t &mem_per_token) {
    const int64_t N = n, n_embd = hp.n_embd, n_head = hp.n_head, n_vocab = hp.n_vocab, hd = n_embd / n_head, past = n_past;
    ggml_context *ctx0 = ggml_init({compute_size, compute_buf.get(), false});
    if (!ctx0) return false;
    ggml_cgraph gf{};
    gf.n_threads = n_threads;
    const size_t es = sizeof(float);

    ggml_tensor *embd = ggml_new_tensor_1d(ctx0, GGML_TYPE_I32, N);
    memcpy(embd->data, tokens, N * sizeof(token_id));
    ggml_tensor *inpL = ggml_get_rows(ctx0, tok_embeddings, embd);
    for (int64_t il = 0; il < hp.n_layer; ++il) {
        const Layer &L = layers[il];
        ggml_tensor *inpSA = inpL;
        ggml_tensor *cur = ggml_rms_norm(ctx0, inpL);
        cur = ggml_mul(ctx0, ggml_repeat(ctx0, L.attention_norm, cur), cur);

        ggml_tensor *Qcur = ggml_rope(ctx0, ggml_reshape_3d(ctx0, ggml_mul_mat(ctx0, L.wq, cur), hd, n_head, N), (int)past, (int)hd, 0);
        ggml_tensor *Kcur = ggml_rope(ctx0, ggml_reshape_3d(ctx0, ggml_mul_mat(ctx0, L.wk, cur), hd, n_head, N), (int)past, (int)hd, 0);
        // this step's K (after rope) and V (transposed: one row per feature) go into the cache
        ggml_tensor *Vcur = ggml_transpose(ctx0, ggml_reshape_2d(ctx0, ggml_mul_mat(ctx0, L.wv, cur), n_embd, N));
        ggml_tensor *kdst = ggml_view_1d(ctx0, k, N * n_embd, es * n_embd * (il * n_ctx + past));
        ggml_tensor *vdst = ggml_view_2d(ctx0, v, N, n_embd, n_ctx * es, il * n_ctx * es * n_embd + past * es);
        ggml_build_forward_expand(&gf, ggml_cpy(ctx0, Kcur, kdst));
        ggml_build_forward_expand(&gf, ggml_cpy(ctx0, Vcur, vdst));

        ggml_tensor *Q = ggml_permute(ctx0, Qcur, 0, 2, 1, 3);
        ggml_tensor *K = ggml_permute(ctx0, ggml_reshape_3d(ctx0, ggml_view_1d(ctx0, k, (past + N) * n_embd, il * n_ctx * es * n_embd), hd, n_head, past + N),
                                      0, 2, 1, 3);
        ggml_tensor *KQ = ggml_mul_mat(ctx0, K, Q);
        ggml_tensor *KQ_scaled = ggml_scale(ctx0, KQ, ggml_new_f32(ctx0, 1.0f / sqrtf(float(n_embd) / n_head)));
        ggml_tensor *KQ_soft_max = ggml_soft_max(ctx0, ggml_diag_mask_inf(ctx0, KQ_scaled, (int)past));
        ggml_tensor *V = ggml_view_3d(ctx0, v, past + N, hd, n_head, n_ctx * es, n_ctx * es * hd, il * n_ctx * es * n_embd);
        ggml_tensor *KQV_merged = ggml_permute(ctx0, ggml_mul_mat(ctx0, V, KQ_soft_max), 0, 2, 1, 3);
        cur = ggml_cpy(ctx0, KQV_merged, ggml_new_tensor_2d(ctx0, GGML_TYPE_F32, n_embd, N));
        cur = ggml_mul_mat(ctx0, L.wo, cur);

        ggml_tensor *inpFF = ggml_add(ctx0, cur, inpSA);
        cur = ggml_rms_norm(ctx0, inpFF);
        cur = ggml_mul(ctx0, ggml_repeat(ctx0, L.ffn_norm, cur), cur);
        ggml_tensor *tmp = ggml_mul_mat(ctx0, L.w3, cur);
        cur = ggml_mul_mat(ctx0, L.w1, cur);
        cur = ggml_mul(ctx0, ggml_silu(ctx0, cur), tmp);
        cur = ggml_mul_mat(ctx0, L.w2, cur);
        inpL = ggml_add(ctx0, cur, inpFF);
    }
    inpL = ggml_rms_norm(ctx0, inpL);
    inpL = ggml_mul(ctx0, ggml_repeat(ctx0, norm, inpL), inpL);
    ggml_tensor *emb = inpL;
    inpL = ggml_mul_mat(ctx0, output, inpL);
    ggml_build_forward_expand(&gf, inpL);
    ggml_graph_compute(ctx0, &gf);

    const float *out = (const float *)ggml_get_data(inpL);
    if (all_logits) {
        logits.assign(out, out + n_vocab * N);
    } else {
        logits.assign(out + n_vocab * (N - 1), out + n_vocab * N);
    }
    if (embeddings_enabled) {
        const float *e = (const float *)ggml_get_data(emb) + n_embd * (N - 1);
        embeddings.assign(e, e + n_embd);
    }
    if (mem_per_token == 0) mem_per_token = ggml_used_mem(ctx0) / N;
    ggml_free(ctx0);
    return true;
}

// ---- sampling ----------------------------------------------------------------------------------------------------------------
// temp <= 0: argmax.  Otherwise: logits / temp with the CTRL repetition penalty on recent tokens, top-k, soft-max, top-p, then one
// draw from std::discrete_distribution (double precision as in fastLLaMa, so a seed gives the same tokens).
token_id sample(const float *logits, int n_vocab, const std::deque<token_id> &recent, double repeat_penalty, int top_k, double top_p, double temp,
                std::mt19937 &rng) {
    if (temp <= 0.0) return (token_id)(std::max_element(logits, logits + n_vocab) - logits);
    const std::unordered_set<token_id> seen(recent.begin(), recent.end());
    std::vector<std::pair<double, token_id>> cand(n_vocab);
    const double scale = 1.0 / temp;
    for (int i = 0; i < n_vocab; ++i) {
        double s = (double)logits[i] * scale;
        if (seen.count(i)) s *= logits[i] < 0.0f ? repeat_penalty : 1.0 / repeat_penalty;
        cand[i] = {s, i};
    }
    const int k = top_k > 0 ? std::min(top_k, n_vocab) : n_vocab;
    std::partial_sort(cand.begin(), cand.begin() + k, cand.end(), [](const auto &a, const auto &b) { return a.first > b.first; });
    cand.resize(k);
    std::vector<double> probs(k);
    double sum = 0.0;
    for (int i = 0; i < k; ++i) {
        probs[i] = (double)std::exp((float)(cand[i].first - cand[0].first));
        sum += probs[i];
    }
    for (double &p : probs) p /= sum;
    if (top_p < 1.0) {
        double cum = 0.0;
        for (size_t i = 0; i < probs.size(); ++i) {
            cum += probs[i];
            if (cum >= top_p) { probs.resize(i + 1); break; }
        }
    }
    std::discrete_distribution<> dist(probs.begin(), probs.end());
    return cand[dist(rng)].second;
}

// ---- session: the state behind one llama_model_context ------------------------------------------------------------------------
template <class T> bool put(FILE *f, const T *p, size_t n = 1) { return fwrite(p, sizeof(T), n, f) == n; }
template <class T> bool get(FILE *f, T *p, size_t n = 1) { return fread(p, sizeof(T), n, f) == n; }

struct Session {
    Log log;
    Model model;
    bool loaded = false;
    int n_past = 0, n_keep = 64, seed = 0;
    size_t last_n_cap = 64, mem_per_token = 0;
    std::mt19937 rng;
    std::vector<token_id> pending;              // tokens accepted but not yet evaluated
    std::deque<token_id> recent;                // the last `last_n_cap` tokens, for the repetition penalty and context recycling
    std::vector<float> logits;
    std::vector<token_id> system_prompt;
    std::vector<std::string> stop_words;
    std::string held_utf8;                      // an incomplete UTF-8 sequence at the end of the streamed text, completed by the next token
    std::string left_over;                      // text after a stop word, streamed at the start of the next generate()

    void remember(token_id t) {
        if (recent.size() >= last_n_cap) recent.pop_front();
        recent.push_back(t);
    }

    // When the pending tokens no longer fit in the context: keep the first n_keep positions and re-evaluate the system prompt and
    // half of the recent tokens after them.
    void recycle_if_full() {
        if (pending.empty() || pending.size() + (size_t)n_past <= (size_t)model.n_ctx) return;
        const size_t remaining = (size_t)(n_past - std::min(n_keep, n_past));
        const size_t n_recent = recent.size() - std::min(remaining >> 1, recent.size());
        n_past = n_keep;
        if (n_recent >= system_prompt.size()) pending.insert(pending.begin(), recent.end() - (std::ptrdiff_t)n_recent, recent.end());
        pending.insert(pending.begin(), system_prompt.begin(), system_prompt.end());
    }

    bool eval_pending() {
        recycle_if_full();
        if (!pending.empty() && !model.eval(n_past, pending.data(), (int)pending.size(), logits, mem_per_token)) return false;
        n_past += (int)pending.size();
        pending.clear();
        return true;
    }

    bool ingest(std::string prompt, bool is_system) {
        log.reset();
        const std::vector<token_id> toks = tokenize(model.vocab, " " + prompt, true);
        if (toks.size() > (size_t)(model.n_ctx - 4)) {
            log.err("ingest", "prompt size(='%zu') exceeds maximum allowed size('%d')", toks.size(), model.n_ctx - 4);
            return false;
        }
        if (is_system) {
            if (n_keep < (int)toks.size()) {
                log.err("ingest", "system prompt size(='%zu') exceeds 'n_keep'(='%d')", toks.size(), n_keep);
                return false;
            }
            system_prompt = toks;
        }
        // every chunk but the last is evaluated here; the last one is evaluated by the next generate() (or ingest())
        const size_t nb = (size_t)model.n_batch;
        for (size_t i = 0; i < toks.size(); i += nb) {
            log.progress(PROGRESS_INGEST, i, toks.size());
            if (!eval_pending()) return false;
            const size_t n = std::min(nb, toks.size() - i);
            pending.assign(toks.begin() + (std::ptrdiff_t)i, toks.begin() + (std::ptrdiff_t)(i + n));
            for (size_t j = 0; j < n; ++j) remember(toks[i + j]);
        }
        log.progress(PROGRESS_INGEST, toks.size(), toks.size());
        recent.clear();
        return true;
    }

    // Streamed text: a trailing incomplete UTF-8 sequence is held back until the next piece completes it.
    void stream(std::string s, llama_stream_fn fn) {
        s = held_utf8 + s;
        held_utf8.clear();
        size_t i = 0, last = 0, n = 0;
        while (i < s.size()) { last = i; n = utf8_len(s[i]); i += n; }
        if (!s.empty() && last + n > s.size()) { held_utf8 = s.substr(last); s.resize(last); }
        if (!s.empty()) fn(s.data(), (int)s.size());
    }

    bool generate(llama_stream_fn fn, size_t n_tokens, int top_k, double top_p, double temp, double repeat_penalty) {
        log.reset();
        // with stop words, up to (longest stop word in tokens) tokens are held back until it is clear they do not start one
        size_t hold = 0;
        for (const auto &w : stop_words) hold = std::max(hold, tokenize(model.vocab, w, false).size());
        if (!left_over.empty()) stream(std::move(left_over), fn);
        left_over.clear();
        std::deque<token_id> held;
        auto flush_one = [&] {
            const token_id t = held.front();
            held.pop_front();
            stream(t >= 0 && t < (token_id)model.vocab.text.size() ? model.vocab.text[t] : std::string(), fn);
        };
        for (size_t step = 0; step < n_tokens; ++step) {
            if (!stop_words.empty()) {
                std::string text = held_utf8;
                for (token_id t : held) text += model.vocab.text[t];
                for (const auto &w : stop_words) {
                    const size_t pos = text.find(w);
                    if (pos == std::string::npos) continue;
                    held_utf8.clear();
                    stream(text.substr(0, pos), fn);
                    left_over = text.substr(pos + w.size());
                    return true;
                }
            }
            if (!eval_pending()) return false;
            const token_id t = sample(logits.data() + logits.size() - model.hp.n_vocab, model.hp.n_vocab, recent, repeat_penalty, top_k, top_p, temp, rng);
            if (t == EOS) break;
            remember(t);
            if (held.size() >= hold && !held.empty()) flush_one();
            held.push_back(t);
            pending.push_back(t);
        }
        while (!held.empty()) flush_one();
        return true;
    }

    // exp(mean negative log-likelihood) of each token given the ones before it, over the second half of every n_batch chunk
    // (each chunk is evaluated from position 0, so every scored token has at least half a chunk of context)
    float perplexity(const char *prompt) {
        const bool old_all = model.all_logits;
        model.all_logits = true;
        const std::vector<token_id> toks = tokenize(model.vocab, prompt, true);
        const size_t nb = (size_t)model.n_batch, nv = (size_t)model.hp.n_vocab;
        double nll = 0.0, res = 0.0;
        size_t count = 0;
        std::vector<float> probs;
        for (size_t i = 0; i < toks.size(); i += nb) {
            const size_t block = std::min(nb, toks.size() - i);
            if (!model.eval(0, toks.data() + i, (int)block, logits, mem_per_token)) { model.all_logits = old_all; return -1.0f; }
            for (size_t j = block / 2; j + 1 < block; ++j) {
                const float *row = logits.data() + j * nv;
                const float mx = *std::max_element(row, row + nv);
                float sum = 0.0f;
                probs.resize(nv);
                for (size_t c = 0; c < nv; ++c) { probs[c] = std::exp(row[c] - mx); sum += probs[c]; }
                nll += (double)-std::log(probs[toks[i + j + 1]] / sum);
                ++count;
            }
            res = std::exp(nll / (double)count);
            log.info("perplexity", "[%zu/%zu]: %.4f\n", i / nb + 1, (toks.size() + nb - 1) / nb, res);
        }
        model.all_logits = old_all;
        return (float)res;
    }

    // State file layout (fastLLaMa's): i32 n_past, u64 + text of the RNG state, u64 mem_per_token, u64 + i32[] pending tokens,
    // u64 + i32[] recent tokens, u64 + f32[] logits, u64 + i32[] system prompt, i32 KV type (f32), K bytes, V bytes.
    bool save_state(const char *path) {
        FILE *f = fopen(path, "wb");
        if (!f) { log.err("save_state", "unable to open '%s'", path); return false; }
        std::stringstream ss;
        ss << rng;
        const std::string r = ss.str();
        const size_t rn = r.size(), np = pending.size(), nr = recent.size(), nl = logits.size(), ns = system_prompt.size();
        const std::vector<token_id> rec(recent.begin(), recent.end());
        const int32_t kv_type = GGML_TYPE_F32;
        // ggml_nbytes on a KV tensor is libggml_b200's cue that the host is about to touch the cache: it brings the device copy back
        const size_t kv_bytes = ggml_nbytes(model.k);
        bool ok = put(f, &n_past) && put(f, &rn) && put(f, r.data(), rn) && put(f, &mem_per_token) && put(f, &np) && put(f, pending.data(), np) &&
                  put(f, &nr) && put(f, rec.data(), nr) && put(f, &nl) && put(f, logits.data(), nl) && put(f, &ns) && put(f, system_prompt.data(), ns) &&
                  put(f, &kv_type) && put(f, (const char *)model.k->data, kv_bytes) && put(f, (const char *)model.v->data, ggml_nbytes(model.v));
        ok = (fclose(f) == 0) && ok;
        if (!ok) log.err("save_state", "writing '%s' failed", path);
        return ok;
    }

    bool load_state(const char *path) {
        FILE *f = fopen(path, "rb");
        if (!f) { log.err("load_state", "unable to open '%s'", path); return false; }
        size_t rn = 0, np = 0, nr = 0, nl = 0, ns = 0;
        int32_t kv_type = -1, np_in = 0;
        const size_t cap = (size_t)model.n_ctx * model.hp.n_vocab + (1u << 20);
        bool ok = get(f, &np_in) && get(f, &rn) && rn < (1u << 20);
        std::string r(ok ? rn : 0, '\0');
        ok = ok && get(f, r.data(), rn) && get(f, &mem_per_token) && get(f, &np) && np <= cap;
        std::vector<token_id> pend(ok ? np : 0);
        ok = ok && get(f, pend.data(), np) && get(f, &nr) && nr <= cap;
        std::vector<token_id> rec(ok ? nr : 0);
        ok = ok && get(f, rec.data(), nr) && get(f, &nl) && nl <= cap;
        std::vector<float> lg(ok ? nl : 0);
        ok = ok && get(f, lg.data(), nl) && get(f, &ns) && ns <= cap;
        std::vector<token_id> sys(ok ? ns : 0);
        ok = ok && get(f, sys.data(), ns) && get(f, &kv_type) && kv_type == GGML_TYPE_F32;
        if (ok) {
            const size_t kv_bytes = ggml_nbytes(model.k);          // (see save_state) the cache is re-uploaded before the next graph
            ok = get(f, (char *)model.k->data, kv_bytes) && get(f, (char *)model.v->data, ggml_nbytes(model.v));
        }
        fclose(f);
        if (!ok) { log.err("load_state", "'%s' is not a state file of this model", path); return false; }
        std::stringstream ss(r);
        ss >> rng;
        n_past = np_in;
        pending = pend;
        recent.assign(rec.begin(), rec.end());
        logits = lg;
        system_prompt = sys;
        return true;
    }

    // ---- LoRA adapters ----
    // An adapter holds, per adapted weight W, either the factors "<W>.loraA" [r, K] and "<W>.loraB" [r, M] (f32, A already
    // scaled by alpha / r) or their product "<W>.lora" [K, M].  Attaching adds B*A to W in place (W's own type: a q4 weight is
    // dequantised, added and re-quantised by ggml_add); detaching subtracts it again.  With a mapped model file W is first copied
    // to private memory, and detaching just points W back at the mapping.
    std::string lora_path;
    std::unique_ptr<uint8_t[]> lora_copies;
    std::unordered_map<std::string, void *> mapped_data;

    bool apply_lora(const std::string &path, bool detach) {
        const char *fn = detach ? "detach_lora" : "attach_lora";
        if (detach && model.use_mmap) {
            for (auto &kv : mapped_data) model.by_name[kv.first]->data = kv.second;
            mapped_data.clear();
            lora_copies.reset();
            lora_path.clear();
            return true;
        }
        FileReader in(path.c_str());
        if (!in.f) { log.err(fn, "failed to open '%s'\n", path.c_str()); return false; }
        uint32_t magic = 0, r = 0, alpha = 0;
        uint8_t cached = 0;
        if (!read_container(in, path.c_str(), log, magic)) return false;
        if (magic != GGLA) { log.err(fn, "'%s' is not a LoRA adapter\n", path.c_str()); return false; }
        std::vector<TensorRecord> dir;
        if (!in.read(cached) || !in.read(r) || !in.read(alpha) || !read_tensor_dir(in, path.c_str(), true, log, dir)) return false;
        if (!detach) log.info(fn, "rank %u, alpha %u, %s\n", r, alpha, cached ? "precomputed B*A" : "factors A and B");

        struct Update { ggml_tensor *base; const TensorRecord *a = nullptr, *b = nullptr; };
        std::vector<std::string> order;
        std::unordered_map<std::string, Update> updates;
        for (const TensorRecord &t : dir) {
            const size_t cut = t.name.rfind(".lora");
            const std::string marker = cut == std::string::npos ? "" : t.name.substr(cut + 5);
            if (cut == std::string::npos || !(cached ? marker.empty() : marker == "A" || marker == "B")) {
                log.err(fn, "'%s' is not a LoRA tensor name\n", t.name.c_str());
                return false;
            }
            const std::string base = t.name.substr(0, cut);
            auto it = model.by_name.find(base);
            if (it == model.by_name.end() || t.ne.size() != 2 || (!cached && t.type != GGML_TYPE_F32)) {
                log.err(fn, "'%s' does not adapt a weight of this model (or is not an f32 matrix)\n", t.name.c_str());
                return false;
            }
            if (!updates.count(base)) order.push_back(base);
            Update &u = updates.emplace(base, Update{it->second}).first->second;
            (marker == "B" ? u.b : u.a) = &t;
        }
        size_t work = 64 * 1024, copies = 0;
        for (auto &kv : updates) {
            Update &u = kv.second;
            const int64_t K = u.base->ne[0], M = u.base->ne[1];
            const bool ok = cached ? (u.a->ne[0] == K && u.a->ne[1] == M)
                                   : (u.a && u.b && u.a->ne[1] == K && u.b->ne[1] == M && u.a->ne[0] == u.b->ne[0]);
            if (!ok) { log.err(fn, "the adapter's matrices for '%s' do not fit its shape\n", kv.first.c_str()); return false; }
            work = std::max(work, (cached ? u.a->size : u.a->size + u.b->size) + 3 * (size_t)(K * M) * sizeof(float) + 64 * 1024);
            copies += ggml_nbytes(u.base);
        }
        if (model.use_mmap) {
            lora_copies.reset(new uint8_t[copies]);
            copies = 0;
        }
        std::unique_ptr<uint8_t[]> buf(new uint8_t[work]);
        auto load = [&](ggml_context *ctx, const TensorRecord &t) -> ggml_tensor * {
            ggml_tensor *x = ggml_new_tensor_2d(ctx, (ggml_type)t.type, t.ne[0], t.ne[1]);
            return fseek(in.f, (long)t.offset, SEEK_SET) == 0 && in.read(x->data, t.size) ? x : nullptr;
        };
        for (const std::string &name : order) {
            Update &u = updates[name];
            if (model.use_mmap) {
                uint8_t *dst = lora_copies.get() + copies;
                copies += ggml_nbytes(u.base);
                memcpy(dst, u.base->data, ggml_nbytes(u.base));
                mapped_data[name] = u.base->data;
                u.base->data = dst;
            }
            ggml_context *ctx = ggml_init({work, buf.get(), false});
            ggml_tensor *a = load(ctx, *u.a), *b = cached ? nullptr : load(ctx, *u.b);
            if (!a || (!cached && !b)) { ggml_free(ctx); log.err(fn, "failed to read '%s'\n", path.c_str()); return false; }
            ggml_tensor *ba = cached ? a : ggml_mul_mat(ctx, a, b);
            if (detach) ba = ggml_scale(ctx, ba, ggml_new_f32(ctx, -1.0f));
            ggml_cgraph gf = ggml_build_forward(ggml_add_inplace(ctx, u.base, ba));
            gf.n_threads = model.n_threads;
            ggml_graph_compute(ctx, &gf);
            ggml_free(ctx);
        }
        lora_path = detach ? std::string() : path;
        return true;
    }

    bool attach_lora(const char *path) {
        if (!lora_path.empty()) { log.err("attach_lora", "'%s' is attached already: detach it first\n", lora_path.c_str()); return false; }
        return apply_lora(path, false);
    }

    bool detach_lora() {
        if (lora_path.empty()) { log.err("detach_lora", "no LoRA adapter is attached\n"); return false; }
        return apply_lora(lora_path, true);
    }

    bool reset() {
        n_past = 0;
        recent.clear();
        logits.clear();
        system_prompt.clear();
        pending.clear();
        rng = std::mt19937((uint32_t)seed);
        model.embeddings.clear();
        return true;
    }
};

}  // namespace

struct llama_model_context {
    llama_model_context_args args;
    std::vector<std::string> stop_words;
    Session *s = nullptr;
    ~llama_model_context() { delete s; }
};

static bool valid(const llama_model_context *c) {
    if (!c) { fprintf(stderr, "model context is not initialised: create one with llama_create_context\n"); return false; }
    if (!c->s) { fprintf(stderr, "no model is loaded: call llama_load_model first\n"); return false; }
    return true;
}

extern "C" {

llama_model_context_args llama_create_default_context_args() {
    llama_model_context_args a{};
    a.seed = 0;
    a.n_keep = 64;
    a.n_ctx = 512;
    a.n_threads = 1;
    a.n_batch = 16;
    a.n_load_parallel_blocks = 1;
    a.last_n_tokens = 64;
    a.logger = {default_info, default_err, default_warn, default_reset, default_progress};
    return a;
}

llama_model_context *llama_create_context(llama_model_context_args args) {
    auto *c = new llama_model_context();
    c->args = args;
    return c;
}

bool llama_load_model(llama_model_context *c, const char *path) {
    if (!c) return false;
    if (c->s) { fprintf(stderr, "a model is already loaded\n"); return false; }
    auto s = std::make_unique<Session>();
    const llama_model_context_args &a = c->args;
    s->log.cb = a.logger;
    s->model.n_ctx = a.n_ctx;
    s->model.n_batch = a.n_batch;
    s->model.n_threads = a.n_threads;
    s->model.use_mmap = a.use_mmap;
    s->model.all_logits = a.should_get_all_logits;
    s->model.embeddings_enabled = a.embedding_eval_enabled;
    s->model.extra_mem = a.allocate_extra_mem;
    s->n_keep = a.n_keep;
    s->seed = a.seed;
    s->rng = std::mt19937((uint32_t)a.seed);
    s->last_n_cap = a.last_n_tokens;
    s->recent.assign(a.last_n_tokens, 0);
    if (a.n_ctx <= 4 || a.n_batch <= 0) { s->log.err("llama_load_model", "n_ctx must exceed 4 and n_batch must be positive\n"); return false; }
    if (!s->model.load(path, s->log)) { s->log.err("llama_load_model", "Unable to load model\n"); return false; }
    c->s = s.release();
    return true;
}

bool llama_set_stop_words(llama_model_context *c, const char **words, size_t n) {
    if (!c) return false;
    c->stop_words.assign(words, words + n);
    return true;
}

bool llama_ingest(llama_model_context *c, const char *prompt) { return valid(c) && c->s->ingest(prompt, false); }
bool llama_ingest_system_prompt(llama_model_context *c, const char *prompt) { return valid(c) && c->s->ingest(prompt, true); }

bool llama_generate(llama_model_context *c, llama_stream_fn fn, size_t n_tokens, float top_k, float top_p, float temp, float repeat_penalty) {
    if (!valid(c)) return false;
    c->s->stop_words = c->stop_words;
    return c->s->generate(fn, n_tokens, (int)top_k, top_p, temp, repeat_penalty);
}

float llama_perplexity(llama_model_context *c, const char *prompt) { return valid(c) ? c->s->perplexity(prompt) : -1.0f; }

llama_array_view_f llama_get_embeddings(const llama_model_context *c) {
    if (!valid(c)) return {nullptr, 0};
    return {c->s->model.embeddings.data(), c->s->model.embeddings.size()};
}

llama_array_view_f llama_get_logits(const llama_model_context *c) {
    if (!valid(c)) return {nullptr, 0};
    return {c->s->logits.data(), c->s->logits.size()};
}

bool llama_save_state(llama_model_context *c, const char *path) { return valid(c) && c->s->save_state(path); }
bool llama_load_state(llama_model_context *c, const char *path) { return valid(c) && c->s->load_state(path); }

bool llama_attach_lora(llama_model_context *c, const char *path) { return valid(c) && c->s->attach_lora(path); }
bool llama_detach_lora(llama_model_context *c) { return valid(c) && c->s->detach_lora(); }

bool llama_reset_model(llama_model_context *c) { return valid(c) && c->s->reset(); }
void llama_free_context(llama_model_context *c) { delete c; }

void llama_handle_signal(int) {
    printf("Quitting the app...");
    exit(0);
}

}  // extern "C"
