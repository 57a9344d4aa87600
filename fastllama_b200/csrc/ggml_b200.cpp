// ggml_b200.cpp -- ggml-compatible host library (boundary B1, include/fl_ggml.h) whose
// ggml_graph_compute runs on a B200 through the extern-"C" CUDA layer (include/fl_cuda.h).
//
// Plain host C++ (compiled by g++, no CUDA headers).  Three parts:
//   1. tensor arena + graph builders: same observable behaviour and space accounting as the
//      reference (reference lib/ggml.c:3666-4075, :4266-5420, :10551-10640), written from scratch;
//   2. device residency: every host arena the graph touches (weights ctx, KV-cache ctx, compute
//      ctx, or a bare mmap'ed range) gets an equally sized device mirror, so a tensor's device
//      address is mirror_base + (tensor->data - arena_base) -- views, KV-slot offsets and reshapes,
//      which ggml encodes purely as host pointer arithmetic, need no translation tables;
//   3. the executor: walks cgraph->nodes in order and issues one or a few kernels per node
//      (replaces ggml_graph_compute + pthread pool + ggml_compute_forward switch,
//      reference lib/ggml.c:10811-11253, :10117-10285).
#include "fl_ggml.h"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "fl_cuda.h"

// ================================================================================================
// small utilities
// ================================================================================================
[[noreturn]] static void b200_abort(const char *file, int line, const char *fmt, ...) {
    fprintf(stderr, "GGML_B200_ASSERT: %s:%d: ", file, line);
    va_list ap;
    va_start(ap, fmt);
    vfprintf(stderr, fmt, ap);
    va_end(ap);
    fprintf(stderr, "\n");
    fflush(stderr);
    abort();
}
#define B200_ASSERT(cond)                                        \
    do {                                                         \
        if (!(cond)) b200_abort(__FILE__, __LINE__, "%s", #cond); \
    } while (0)
#define B200_FAIL(...) b200_abort(__FILE__, __LINE__, __VA_ARGS__)
// every call into the CUDA layer is checked; a failure is fatal (like GGML_ASSERT -> abort())
#define FLC(expr)                                                                                 \
    do {                                                                                          \
        if ((expr) != 0) b200_abort(__FILE__, __LINE__, "%s failed: %s", #expr, fl_last_error()); \
    } while (0)

static const int k_blck[GGML_TYPE_COUNT] = {1, 1, 32, 32, 16, 16, 32, 1, 1, 1};
static const size_t k_tsize[GGML_TYPE_COUNT] = {4, 2, 20, 24, 10, 12, 40, 1, 2, 4};
static const char *k_tname[GGML_TYPE_COUNT] = {"f32", "f16", "q4_0", "q4_1", "q4_2", "q4_3", "q8_0", "i8", "i16", "i32"};
static const char *k_opname[GGML_OP_COUNT] = {
    "NONE", "DUP", "ADD", "SUB", "MUL", "DIV", "SQR", "SQRT", "SUM", "MEAN", "REPEAT", "ABS", "SGN", "NEG", "STEP",
    "RELU", "GELU", "SILU", "NORM", "RMS_NORM", "MUL_MAT", "SCALE", "CPY", "CONT", "RESHAPE", "VIEW", "PERMUTE",
    "TRANSPOSE", "GET_ROWS", "DIAG_MASK_INF", "SOFT_MAX", "ROPE", "CONV_1D_1S", "CONV_1D_2S", "FLASH_ATTN", "FLASH_FF",
    "MAP_UNARY", "MAP_BINARY"};
static constexpr size_t MEM_ALIGN = 16;

extern "C" {

void ggml_time_init(void) {}
int64_t ggml_time_us(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (int64_t)ts.tv_sec * 1000000 + (int64_t)ts.tv_nsec / 1000;
}
int64_t ggml_time_ms(void) { return ggml_time_us() / 1000; }

// IEEE binary16 <-> binary32, round-to-nearest-even (what _cvtss_sh / _cvtsh_ss do)
float ggml_fp16_to_fp32(ggml_fp16_t h) {
    const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
    uint32_t exp = (h >> 10) & 0x1Fu, man = h & 0x3FFu, bits;
    if (exp == 0) {
        if (man == 0) bits = sign;
        else {
            int e = -1;
            do { e++; man <<= 1; } while ((man & 0x400u) == 0);
            bits = sign | ((uint32_t)(127 - 15 - e) << 23) | ((man & 0x3FFu) << 13);
        }
    } else if (exp == 31) bits = sign | 0x7F800000u | (man << 13);
    else bits = sign | ((exp + 112u) << 23) | (man << 13);
    float f;
    memcpy(&f, &bits, 4);
    return f;
}
ggml_fp16_t ggml_fp32_to_fp16(float f) {
    uint32_t x;
    memcpy(&x, &f, 4);
    const uint32_t sign = (x >> 16) & 0x8000u;
    const uint32_t ax = x & 0x7FFFFFFFu;
    if (ax >= 0x7F800000u) return (ggml_fp16_t)(sign | 0x7C00u | (ax > 0x7F800000u ? 0x200u | ((ax >> 13) & 0x3FFu) : 0u));
    if (ax >= 0x477FF000u) return (ggml_fp16_t)(sign | 0x7C00u);               // rounds to inf
    if (ax < 0x33000001u) return (ggml_fp16_t)sign;                             // rounds to zero
    int e = (int)(ax >> 23) - 127;
    uint32_t man = (ax & 0x7FFFFFu) | 0x800000u;
    uint32_t shift, hexp;
    if (e < -14) { shift = (uint32_t)(13 + (-14 - e)); hexp = 0; }
    else         { shift = 13; hexp = (uint32_t)(e + 15); }
    uint32_t hman = man >> shift;
    const uint32_t rem = man & ((1u << shift) - 1u), half = 1u << (shift - 1);
    if (rem > half || (rem == half && (hman & 1u))) hman++;
    uint32_t out = (e < -14) ? hman : (((hexp << 10) | (hman & 0x3FFu)) + ((hman & 0x800u) ? 0x400u : 0u));
    if (e >= -14 && (hman & 0x800u)) out = ((hexp + 1) << 10);                  // mantissa overflow
    return (ggml_fp16_t)(sign | out);
}

int ggml_cpu_has_blas(void) { return 0; }
int ggml_cpu_has_cublas(void) { return 0; }

int64_t ggml_nelements(const struct ggml_tensor *t) { return t->ne[0] * t->ne[1] * t->ne[2] * t->ne[3]; }
static inline size_t nbytes_of(const struct ggml_tensor *t) { return (size_t)(ggml_nelements(t) * (int64_t)k_tsize[t->type]) / k_blck[t->type]; }
static void host_access_hook(const struct ggml_tensor *t);
// number of persistent arenas the device has written since their last host sync: while it is zero the exported ggml_nbytes is a pure
// function (the reference's loader calls it from several threads, include/file_loader.hpp load_parallel)
static std::atomic<int> g_dirty_arenas{0};
// Exported ggml_nbytes doubles as the host-access hook of device-written arenas: see host_access_hook below.
size_t ggml_nbytes(const struct ggml_tensor *t) {
    if (g_dirty_arenas.load(std::memory_order_acquire) != 0) host_access_hook(t);
    return nbytes_of(t);
}
int ggml_blck_size(enum ggml_type type) { return k_blck[type]; }
size_t ggml_type_size(enum ggml_type type) { return k_tsize[type]; }
float ggml_type_sizef(enum ggml_type type) { return (float)k_tsize[type] / k_blck[type]; }
const char *ggml_type_name(enum ggml_type type) { return k_tname[type]; }
size_t ggml_element_size(const struct ggml_tensor *t) { return k_tsize[t->type]; }
bool ggml_is_quantized(enum ggml_type type) { return type >= GGML_TYPE_Q4_0 && type <= GGML_TYPE_Q8_0; }

}  // extern "C"

static inline int64_t nrows(const ggml_tensor *t) { return t->ne[1] * t->ne[2] * t->ne[3]; }
static inline bool same_shape(const ggml_tensor *a, const ggml_tensor *b) {
    return a->ne[0] == b->ne[0] && a->ne[1] == b->ne[1] && a->ne[2] == b->ne[2] && a->ne[3] == b->ne[3];
}
static inline bool is_contiguous(const ggml_tensor *t) {
    return t->nb[0] == k_tsize[t->type] && t->nb[1] == (t->nb[0] * t->ne[0]) / k_blck[t->type] &&
           t->nb[2] == t->nb[1] * t->ne[1] && t->nb[3] == t->nb[2] * t->ne[2];
}

// ================================================================================================
// 1. contexts: a pool of 64 bump arenas over caller-provided (or owned) buffers
// ================================================================================================
struct ggml_context {
    size_t mem_size;
    char *mem_buffer;
    bool owned, no_alloc;
    int n_objects;
    ggml_object *first, *last;
    ggml_scratch scratch, scratch_save;
    int mirror_id;            // index of this arena's device mirror record
};
namespace {
struct Slot { bool used; ggml_context ctx; };
Slot g_slots[GGML_MAX_CONTEXTS];
}  // namespace
static void mirrors_on_ctx_init(ggml_context *ctx);
static void mirrors_on_ctx_free(ggml_context *ctx);
static void mirrors_on_scratch(void *data, size_t size);
static void mirrors_note_alloc(ggml_context *ctx, size_t end);

extern "C" struct ggml_context *ggml_init(struct ggml_init_params params) {
    for (auto &slot : g_slots) {
        if (slot.used) continue;
        slot.used = true;
        ggml_context *c = &slot.ctx;
        memset(c, 0, sizeof(*c));
        c->mem_size = (params.mem_size + MEM_ALIGN - 1) & ~(MEM_ALIGN - 1);
        c->owned = params.mem_buffer == nullptr;
        c->mem_buffer = c->owned ? (char *)aligned_alloc(MEM_ALIGN, c->mem_size ? c->mem_size : MEM_ALIGN) : (char *)params.mem_buffer;
        c->no_alloc = params.no_alloc;
        B200_ASSERT(c->mem_buffer != nullptr);
        B200_ASSERT(((uintptr_t)c->mem_buffer % MEM_ALIGN) == 0);
        mirrors_on_ctx_init(c);
        return c;
    }
    return nullptr;
}

extern "C" void ggml_free(struct ggml_context *ctx) {
    for (auto &slot : g_slots) {
        if (&slot.ctx != ctx) continue;
        mirrors_on_ctx_free(ctx);
        if (ctx->owned) free(ctx->mem_buffer);
        slot.used = false;
        return;
    }
}

extern "C" size_t ggml_used_mem(const struct ggml_context *ctx) { return ctx->last ? ctx->last->offs + ctx->last->size : 0; }

extern "C" size_t ggml_set_scratch(struct ggml_context *ctx, struct ggml_scratch scratch) {
    const size_t prev = ctx->scratch.data ? ctx->scratch.offs : 0;
    ctx->scratch = scratch;
    if (scratch.data) mirrors_on_scratch(scratch.data, scratch.size);
    return prev;
}

// Space accounting follows the reference bump allocator exactly (lib/ggml.c:3809-3928): an object
// header, then the tensor struct, then (unless the data lives elsewhere) the payload rounded up to
// 16 bytes; with a scratch buffer active the payload goes to the scratch arena instead.
static ggml_tensor *new_tensor_impl(ggml_context *ctx, ggml_type type, int n_dims, const int64_t *ne, void *data) {
    const size_t cur_end = ctx->last ? ctx->last->offs + ctx->last->size : 0;
    size_t payload = 0;
    if (data == nullptr && !ctx->no_alloc) {
        payload = k_tsize[type] * (size_t)(ne[0] / k_blck[type]);
        for (int i = 1; i < n_dims; i++) payload *= (size_t)ne[i];
        payload = (payload + MEM_ALIGN - 1) / MEM_ALIGN * MEM_ALIGN;
    }
    ggml_object *obj = (ggml_object *)(ctx->mem_buffer + cur_end);
    size_t obj_size;
    if (ctx->scratch.data == nullptr || data != nullptr) {
        obj_size = payload + sizeof(ggml_tensor);
        if (cur_end + obj_size + sizeof(ggml_object) > ctx->mem_size) {
            fprintf(stderr, "ggml_new_tensor_impl: not enough space in the context's memory pool (needed %zu, available %zu)\n",
                    cur_end + obj_size + sizeof(ggml_object), ctx->mem_size);
            return nullptr;
        }
    } else {
        if (ctx->scratch.offs + payload > ctx->scratch.size) {
            fprintf(stderr, "ggml_new_tensor_impl: not enough space in the scratch memory\n");
            return nullptr;
        }
        obj_size = sizeof(ggml_tensor);
        if (cur_end + obj_size + sizeof(ggml_object) > ctx->mem_size) {
            fprintf(stderr, "ggml_new_tensor_impl: not enough space in the context's memory pool\n");
            return nullptr;
        }
        data = (char *)ctx->scratch.data + ctx->scratch.offs;
        ctx->scratch.offs += payload;
    }
    obj->offs = cur_end + sizeof(ggml_object);
    obj->size = obj_size;
    obj->next = nullptr;
    if (ctx->last) ctx->last->next = obj; else ctx->first = obj;
    ctx->last = obj;
    ctx->n_objects++;
    mirrors_note_alloc(ctx, obj->offs + obj->size);

    ggml_tensor *t = (ggml_tensor *)(ctx->mem_buffer + obj->offs);
    memset(t, 0, sizeof(*t));
    t->type = type;
    t->n_dims = n_dims;
    for (int i = 0; i < GGML_MAX_DIMS; i++) t->ne[i] = i < n_dims ? ne[i] : 1;
    t->nb[0] = k_tsize[type];
    t->nb[1] = t->nb[0] * (size_t)(t->ne[0] / k_blck[type]);
    for (int i = 2; i < GGML_MAX_DIMS; i++) t->nb[i] = t->nb[i - 1] * (size_t)t->ne[i - 1];
    t->op = GGML_OP_NONE;
    t->data = (data == nullptr && !ctx->no_alloc) ? (void *)(t + 1) : data;
    return t;
}

extern "C" {
struct ggml_tensor *ggml_new_tensor(struct ggml_context *ctx, enum ggml_type type, int n_dims, const int64_t *ne) {
    return new_tensor_impl(ctx, type, n_dims, ne, nullptr);
}
struct ggml_tensor *ggml_new_tensor_1d(struct ggml_context *ctx, enum ggml_type type, int64_t ne0) {
    return new_tensor_impl(ctx, type, 1, &ne0, nullptr);
}
struct ggml_tensor *ggml_new_tensor_2d(struct ggml_context *ctx, enum ggml_type type, int64_t ne0, int64_t ne1) {
    const int64_t ne[2] = {ne0, ne1};
    return new_tensor_impl(ctx, type, 2, ne, nullptr);
}
struct ggml_tensor *ggml_new_tensor_3d(struct ggml_context *ctx, enum ggml_type type, int64_t ne0, int64_t ne1, int64_t ne2) {
    const int64_t ne[3] = {ne0, ne1, ne2};
    return new_tensor_impl(ctx, type, 3, ne, nullptr);
}
struct ggml_tensor *ggml_new_tensor_4d(struct ggml_context *ctx, enum ggml_type type, int64_t ne0, int64_t ne1, int64_t ne2, int64_t ne3) {
    const int64_t ne[4] = {ne0, ne1, ne2, ne3};
    return new_tensor_impl(ctx, type, 4, ne, nullptr);
}
// scalar constants never go to the scratch arena (reference lib/ggml.c:3978-4003)
struct ggml_tensor *ggml_new_i32(struct ggml_context *ctx, int32_t value) {
    ctx->scratch_save = ctx->scratch;
    ctx->scratch.data = nullptr;
    ggml_tensor *t = ggml_new_tensor_1d(ctx, GGML_TYPE_I32, 1);
    ctx->scratch = ctx->scratch_save;
    *(int32_t *)t->data = value;
    return t;
}
struct ggml_tensor *ggml_new_f32(struct ggml_context *ctx, float value) {
    ctx->scratch_save = ctx->scratch;
    ctx->scratch.data = nullptr;
    ggml_tensor *t = ggml_new_tensor_1d(ctx, GGML_TYPE_F32, 1);
    ctx->scratch = ctx->scratch_save;
    *(float *)t->data = value;
    return t;
}
struct ggml_tensor *ggml_dup_tensor(struct ggml_context *ctx, const struct ggml_tensor *src) {
    return new_tensor_impl(ctx, src->type, src->n_dims, src->ne, nullptr);
}
struct ggml_tensor *ggml_view_tensor(struct ggml_context *ctx, const struct ggml_tensor *src) {
    ggml_tensor *t = new_tensor_impl(ctx, src->type, src->n_dims, src->ne, src->data);
    for (int i = 0; i < GGML_MAX_DIMS; i++) t->nb[i] = src->nb[i];
    return t;
}
struct ggml_tensor *ggml_set_zero(struct ggml_tensor *t) {
    memset(t->data, 0, nbytes_of(t));
    return t;
}
struct ggml_tensor *ggml_set_i32(struct ggml_tensor *t, int32_t value) {
    const int64_t n = ggml_nelements(t);
    B200_ASSERT(is_contiguous(t));
    switch (t->type) {
        case GGML_TYPE_I8:  for (int64_t i = 0; i < n; i++) ((int8_t *)t->data)[i] = (int8_t)value; break;
        case GGML_TYPE_I16: for (int64_t i = 0; i < n; i++) ((int16_t *)t->data)[i] = (int16_t)value; break;
        case GGML_TYPE_I32: for (int64_t i = 0; i < n; i++) ((int32_t *)t->data)[i] = value; break;
        case GGML_TYPE_F16: for (int64_t i = 0; i < n; i++) ((ggml_fp16_t *)t->data)[i] = ggml_fp32_to_fp16((float)value); break;
        case GGML_TYPE_F32: for (int64_t i = 0; i < n; i++) ((float *)t->data)[i] = (float)value; break;
        default: B200_FAIL("ggml_set_i32: unsupported type %s", k_tname[t->type]);
    }
    return t;
}
struct ggml_tensor *ggml_set_f32(struct ggml_tensor *t, float value) {
    const int64_t n = ggml_nelements(t);
    B200_ASSERT(is_contiguous(t));
    switch (t->type) {
        case GGML_TYPE_I8:  for (int64_t i = 0; i < n; i++) ((int8_t *)t->data)[i] = (int8_t)value; break;
        case GGML_TYPE_I16: for (int64_t i = 0; i < n; i++) ((int16_t *)t->data)[i] = (int16_t)value; break;
        case GGML_TYPE_I32: for (int64_t i = 0; i < n; i++) ((int32_t *)t->data)[i] = (int32_t)value; break;
        case GGML_TYPE_F16: for (int64_t i = 0; i < n; i++) ((ggml_fp16_t *)t->data)[i] = ggml_fp32_to_fp16(value); break;
        case GGML_TYPE_F32: for (int64_t i = 0; i < n; i++) ((float *)t->data)[i] = value; break;
        default: B200_FAIL("ggml_set_f32: unsupported type %s", k_tname[t->type]);
    }
    return t;
}
void *ggml_get_data(const struct ggml_tensor *t) { return t->data; }
float *ggml_get_data_f32(const struct ggml_tensor *t) { return (float *)t->data; }

// ================================================================================================
// graph builders (host only).  Inference graphs carry no gradients, so ->grad stays NULL.
// ================================================================================================
static ggml_tensor *op_node(ggml_tensor *res, ggml_op op, ggml_tensor *a, ggml_tensor *b) {
    res->op = op;
    res->src0 = a;
    res->src1 = b;
    return res;
}
#define NO_GRAD(t) B200_ASSERT((t) == nullptr || (t)->grad == nullptr)

struct ggml_tensor *ggml_dup(struct ggml_context *ctx, struct ggml_tensor *a) {
    NO_GRAD(a);
    return op_node(ggml_dup_tensor(ctx, a), GGML_OP_DUP, a, nullptr);
}
struct ggml_tensor *ggml_add(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    NO_GRAD(a); NO_GRAD(b);
    B200_ASSERT(same_shape(a, b));
    return op_node(ggml_dup_tensor(ctx, a), GGML_OP_ADD, a, b);
}
struct ggml_tensor *ggml_add_inplace(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    B200_ASSERT(same_shape(a, b));
    return op_node(ggml_view_tensor(ctx, a), GGML_OP_ADD, a, b);
}
struct ggml_tensor *ggml_mul(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    NO_GRAD(a); NO_GRAD(b);
    B200_ASSERT(same_shape(a, b));
    return op_node(ggml_dup_tensor(ctx, a), GGML_OP_MUL, a, b);
}
struct ggml_tensor *ggml_repeat(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    NO_GRAD(a);
    B200_ASSERT(b->ne[0] % a->ne[0] == 0 && b->ne[1] % a->ne[1] == 0 && b->ne[2] % a->ne[2] == 0 && b->ne[3] % a->ne[3] == 0);
    if (same_shape(a, b)) return a;      // reference lib/ggml.c:4602-4604
    return op_node(ggml_new_tensor(ctx, a->type, b->n_dims, b->ne), GGML_OP_REPEAT, a, b);
}
struct ggml_tensor *ggml_silu(struct ggml_context *ctx, struct ggml_tensor *a) {
    NO_GRAD(a);
    return op_node(ggml_dup_tensor(ctx, a), GGML_OP_SILU, a, nullptr);
}
struct ggml_tensor *ggml_rms_norm(struct ggml_context *ctx, struct ggml_tensor *a) {
    NO_GRAD(a);
    return op_node(ggml_dup_tensor(ctx, a), GGML_OP_RMS_NORM, a, nullptr);
}
struct ggml_tensor *ggml_mul_mat(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    NO_GRAD(a); NO_GRAD(b);
    B200_ASSERT(a->ne[0] == b->ne[0] && a->ne[2] == b->ne[2] && a->ne[3] == b->ne[3]);   // ggml_can_mul_mat
    B200_ASSERT(a->nb[0] <= a->nb[1]);                                                    // !ggml_is_transposed(a)
    const int64_t ne[4] = {a->ne[1], b->ne[1], a->ne[2], b->ne[3]};
    return op_node(ggml_new_tensor(ctx, GGML_TYPE_F32, std::min(a->n_dims, b->n_dims), ne), GGML_OP_MUL_MAT, a, b);
}
struct ggml_tensor *ggml_scale(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    NO_GRAD(a); NO_GRAD(b);
    B200_ASSERT(ggml_nelements(b) == 1);
    return op_node(ggml_view_tensor(ctx, a), GGML_OP_SCALE, a, b);          // in place, returns view(a)
}
struct ggml_tensor *ggml_cpy(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    NO_GRAD(a); NO_GRAD(b);
    B200_ASSERT(ggml_nelements(a) == ggml_nelements(b));
    return op_node(ggml_view_tensor(ctx, b), GGML_OP_CPY, a, b);            // result is a view of the destination
}
struct ggml_tensor *ggml_cont(struct ggml_context *ctx, struct ggml_tensor *a) {
    NO_GRAD(a);
    return op_node(ggml_dup_tensor(ctx, a), GGML_OP_CONT, a, nullptr);
}
struct ggml_tensor *ggml_reshape(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    NO_GRAD(a);
    B200_ASSERT(is_contiguous(a) && is_contiguous(b) && ggml_nelements(a) == ggml_nelements(b));
    return op_node(new_tensor_impl(ctx, a->type, b->n_dims, b->ne, a->data), GGML_OP_RESHAPE, a, nullptr);
}
struct ggml_tensor *ggml_reshape_2d(struct ggml_context *ctx, struct ggml_tensor *a, int64_t ne0, int64_t ne1) {
    NO_GRAD(a);
    B200_ASSERT(is_contiguous(a) && ggml_nelements(a) == ne0 * ne1);
    const int64_t ne[2] = {ne0, ne1};
    return op_node(new_tensor_impl(ctx, a->type, 2, ne, a->data), GGML_OP_RESHAPE, a, nullptr);
}
struct ggml_tensor *ggml_reshape_3d(struct ggml_context *ctx, struct ggml_tensor *a, int64_t ne0, int64_t ne1, int64_t ne2) {
    NO_GRAD(a);
    B200_ASSERT(is_contiguous(a) && ggml_nelements(a) == ne0 * ne1 * ne2);
    const int64_t ne[3] = {ne0, ne1, ne2};
    return op_node(new_tensor_impl(ctx, a->type, 3, ne, a->data), GGML_OP_RESHAPE, a, nullptr);
}
struct ggml_tensor *ggml_view_1d(struct ggml_context *ctx, struct ggml_tensor *a, int64_t ne0, size_t offset) {
    NO_GRAD(a);
    return op_node(new_tensor_impl(ctx, a->type, 1, &ne0, (char *)a->data + offset), GGML_OP_VIEW, a, nullptr);
}
struct ggml_tensor *ggml_view_2d(struct ggml_context *ctx, struct ggml_tensor *a, int64_t ne0, int64_t ne1, size_t nb1, size_t offset) {
    NO_GRAD(a);
    const int64_t ne[2] = {ne0, ne1};
    ggml_tensor *t = new_tensor_impl(ctx, a->type, 2, ne, (char *)a->data + offset);
    t->nb[1] = nb1;
    t->nb[2] = t->nb[1] * (size_t)ne1;
    t->nb[3] = t->nb[2];
    return op_node(t, GGML_OP_VIEW, a, nullptr);
}
struct ggml_tensor *ggml_view_3d(struct ggml_context *ctx, struct ggml_tensor *a, int64_t ne0, int64_t ne1, int64_t ne2, size_t nb1, size_t nb2, size_t offset) {
    NO_GRAD(a);
    const int64_t ne[3] = {ne0, ne1, ne2};
    ggml_tensor *t = new_tensor_impl(ctx, a->type, 3, ne, (char *)a->data + offset);
    t->nb[1] = nb1;
    t->nb[2] = nb2;
    t->nb[3] = t->nb[2] * (size_t)ne2;
    return op_node(t, GGML_OP_VIEW, a, nullptr);
}
struct ggml_tensor *ggml_permute(struct ggml_context *ctx, struct ggml_tensor *a, int ax0, int ax1, int ax2, int ax3) {
    NO_GRAD(a);
    const int ax[4] = {ax0, ax1, ax2, ax3};
    bool seen[4] = {false, false, false, false};
    for (int i = 0; i < 4; i++) {
        B200_ASSERT(ax[i] >= 0 && ax[i] < 4 && !seen[ax[i]]);
        seen[ax[i]] = true;
    }
    ggml_tensor *t = ggml_view_tensor(ctx, a);
    for (int i = 0; i < 4; i++) {       // source axis i becomes axis ax[i]
        t->ne[ax[i]] = a->ne[i];
        t->nb[ax[i]] = a->nb[i];
    }
    return op_node(t, GGML_OP_PERMUTE, a, nullptr);
}
struct ggml_tensor *ggml_transpose(struct ggml_context *ctx, struct ggml_tensor *a) {
    NO_GRAD(a);
    ggml_tensor *t = ggml_view_tensor(ctx, a);
    t->ne[0] = a->ne[1]; t->ne[1] = a->ne[0];
    t->nb[0] = a->nb[1]; t->nb[1] = a->nb[0];
    return op_node(t, GGML_OP_TRANSPOSE, a, nullptr);
}
struct ggml_tensor *ggml_get_rows(struct ggml_context *ctx, struct ggml_tensor *a, struct ggml_tensor *b) {
    NO_GRAD(a); NO_GRAD(b);
    B200_ASSERT(a->ne[2] == 1 && a->ne[3] == 1 && b->ne[1] == 1 && b->ne[2] == 1 && b->ne[3] == 1 && b->type == GGML_TYPE_I32);
    return op_node(ggml_new_tensor_2d(ctx, GGML_TYPE_F32, a->ne[0], b->ne[0]), GGML_OP_GET_ROWS, a, b);
}
struct ggml_tensor *ggml_diag_mask_inf(struct ggml_context *ctx, struct ggml_tensor *a, int n_past) {
    NO_GRAD(a);
    ggml_tensor *t = ggml_view_tensor(ctx, a);
    ggml_tensor *p = ggml_new_i32(ctx, n_past);
    return op_node(t, GGML_OP_DIAG_MASK_INF, a, p);
}
struct ggml_tensor *ggml_soft_max(struct ggml_context *ctx, struct ggml_tensor *a) {
    NO_GRAD(a);
    return op_node(ggml_view_tensor(ctx, a), GGML_OP_SOFT_MAX, a, nullptr);
}
struct ggml_tensor *ggml_rope(struct ggml_context *ctx, struct ggml_tensor *a, int n_past, int n_dims, int mode) {
    NO_GRAD(a);
    B200_ASSERT(n_past >= 0);
    ggml_tensor *t = ggml_view_tensor(ctx, a);
    ggml_tensor *p = ggml_new_tensor_1d(ctx, GGML_TYPE_I32, 3);
    ((int32_t *)p->data)[0] = n_past;
    ((int32_t *)p->data)[1] = n_dims;
    ((int32_t *)p->data)[2] = mode;
    return op_node(t, GGML_OP_ROPE, a, p);
}
}  // extern "C"

// ------------------------------------------------------------------------------------------------
// graph construction: depth-first post-order like the reference (lib/ggml.c:10551-10600) so node
// order -- and therefore execution order on the stream -- is identical.  The reference finds
// "already visited" by scanning the node list (O(n^2), ~0.4 ms for a 7B graph); we stamp each
// tensor's spare padding bytes with (graph epoch, index) instead.
// ------------------------------------------------------------------------------------------------
namespace {
struct Stamp { uint32_t epoch; int32_t index; };     // lives in ggml_tensor::padding (8 bytes)
static_assert(sizeof(Stamp) == 8, "stamp must fit the tensor padding");
uint32_t g_epoch = 0;                                // last epoch handed out
// Which epoch a cgraph's stamps carry.  `clean` = every tensor of the graph was stamped under this
// entry (false for a graph we first meet half-built, e.g. a by-value copy of ggml_build_forward's
// result): then membership falls back to the reference's pointer scan.
struct GraphEpoch { const ggml_cgraph *g; uint32_t epoch; bool clean; };
GraphEpoch g_graph_epochs[8];
int g_graph_epoch_next = 0;

inline Stamp *stamp_of(ggml_tensor *t) { return (Stamp *)t->padding; }

GraphEpoch *lookup_epoch(const ggml_cgraph *g) {
    for (auto &ge : g_graph_epochs)
        if (ge.g == g && ge.epoch != 0) return &ge;
    return nullptr;
}
GraphEpoch *new_epoch(const ggml_cgraph *g, bool clean) {
    if (++g_epoch == 0) ++g_epoch;
    GraphEpoch *slot = lookup_epoch(g);
    if (!slot) {
        slot = &g_graph_epochs[g_graph_epoch_next];
        g_graph_epoch_next = (g_graph_epoch_next + 1) % 8;
    }
    *slot = GraphEpoch{g, g_epoch, clean};
    return slot;
}

// index encoding: >= 0 node index, < 0 -> leaf index = -1 - index
bool graph_contains(const ggml_cgraph *g, const ggml_tensor *t, uint32_t epoch, bool interleaved) {
    const Stamp *s = (const Stamp *)t->padding;
    if (s->epoch == epoch) {
        if (s->index >= 0 && s->index < g->n_nodes && g->nodes[s->index] == t) return true;
        if (s->index < 0 && -1 - s->index < g->n_leafs && g->leafs[-1 - s->index] == t) return true;
    }
    if (!interleaved) return false;
    for (int i = 0; i < g->n_nodes; i++) if (g->nodes[i] == t) return true;     // another graph re-stamped it
    for (int i = 0; i < g->n_leafs; i++) if (g->leafs[i] == t) return true;
    return false;
}

void visit(ggml_cgraph *g, ggml_tensor *t, uint32_t epoch, bool interleaved) {
    if (graph_contains(g, t, epoch, interleaved)) return;
    if (t->src0) visit(g, t->src0, epoch, interleaved);
    if (t->src1) visit(g, t->src1, epoch, interleaved);
    for (int i = 0; i < GGML_MAX_OPT; i++) if (t->opt[i]) visit(g, t->opt[i], epoch, interleaved);
    Stamp *s = stamp_of(t);
    if (t->op == GGML_OP_NONE && t->grad == nullptr) {
        B200_ASSERT(g->n_leafs < GGML_MAX_NODES);
        s->epoch = epoch; s->index = -1 - g->n_leafs;
        g->leafs[g->n_leafs++] = t;
    } else {
        B200_ASSERT(g->n_nodes < GGML_MAX_NODES);
        s->epoch = epoch; s->index = g->n_nodes;
        g->grads[g->n_nodes] = t->grad;
        g->nodes[g->n_nodes++] = t;
    }
}
}  // namespace

extern "C" void ggml_build_forward_expand(struct ggml_cgraph *g, struct ggml_tensor *tensor) {
    const bool fresh = g->n_nodes == 0 && g->n_leafs == 0;
    GraphEpoch *ge = fresh ? new_epoch(g, true) : lookup_epoch(g);
    if (!ge) ge = new_epoch(g, false);
    // stamps are authoritative only while no other graph has been started since (it may have
    // re-stamped shared tensors such as weights) and the graph was stamped from its first node
    const bool scan = !ge->clean || ge->epoch != g_epoch;
    const int n0 = g->n_nodes;
    visit(g, tensor, ge->epoch, scan);
    if (g->n_nodes > n0) B200_ASSERT(g->nodes[g->n_nodes - 1] == tensor);
}
extern "C" struct ggml_cgraph ggml_build_forward(struct ggml_tensor *tensor) {
    static thread_local ggml_cgraph g;               // returned by value; the static avoids a 96 KB stack temp
    memset(&g, 0, sizeof(g));
    g.n_threads = GGML_DEFAULT_N_THREADS;
    // build into the static, then re-key the epoch entry so the caller's copy keeps working
    ggml_build_forward_expand(&g, tensor);
    return g;
}

// ================================================================================================
// 2. device residency: mirrors of host arenas
// ================================================================================================
namespace {
enum MirrorKind { MK_ARENA = 0, MK_EXTERNAL = 1, MK_SCRATCH = 2 };
// The reference wraps every ggml_context in an RAII type whose defaulted move leaves the pointer in
// the moved-from temporary, so contexts are "freed" right after they are created and their pool
// slots are re-used (reference include/tensor/mem_context.hpp:31-43) -- harmless there because
// ggml_free only releases the slot.  Mirrors are therefore keyed by the ARENA (host range), never
// by context identity or lifetime; how far an arena has been filled is recorded by the allocator.
struct Mirror {
    const char *host;        // arena base
    size_t size;
    char *dev;               // equally sized device allocation (lazy)
    size_t alloc_end;        // bytes of the arena handed out by the bump allocator so far
    size_t uploaded;         // bytes [0, uploaded) of a persistent arena already copied to the device
    int kind;                // MK_ARENA: a ggml context buffer; MK_EXTERNAL: a bare tensor range that is
                             // not a ggml arena (mmap'ed weights), uploaded once; MK_SCRATCH: a
                             // ggml_set_scratch buffer (activations only, never uploaded)
    bool alive;
    bool device_dirty = false;   // a graph wrote into this persistent arena on the device (KV cache) since the last host sync
};
std::vector<Mirror> g_mirrors;
int g_last_mirror = -1;
bool g_verbose = false;

struct Stats { uint64_t n_evals = 0; double last_us = 0, total_us = 0; uint64_t graph_replays = 0; } g_stats;
// host-side time of the fused decode path, microseconds summed over decode steps (ggml_b200_get_host_profile):
// [0] steps, [1] graph match, [2] scalars + launch issue, [3] waiting for the device + result copies, [4] between two graph computes (caller:
// sampling, graph building, callbacks)
double g_hostprof[8] = {0, 0, 0, 0, 0, 0, 0, 0};
int64_t g_last_exit_us = 0;
bool g_profile = false;
int g_decode_mode = 0;          // see ggml_b200_decode_mode()
bool g_tp_kv_sharded = false;   // tensor-parallel decode steps have written only this rank's heads into the KV cache
std::vector<ggml_b200_kernel_stat> g_kstats;
void *g_pev0 = nullptr, *g_pev1 = nullptr;

void ensure_backend() {
    static bool done = false;
    if (done) return;
    if (fl_init(-1) != 0) B200_FAIL("cannot initialise the B200 backend: %s", fl_last_error());
    g_verbose = getenv("FASTLLAMA_B200_VERBOSE") != nullptr;
    done = true;
}

void drop_mirror(Mirror &m) {
    if (m.device_dirty) { m.device_dirty = false; g_dirty_arenas.fetch_sub(1, std::memory_order_release); }
    if (m.dev) {
        if (fl_is_initialized()) fl_dev_free(m.dev);
        m.dev = nullptr;
    }
}

int find_mirror(const void *p) {
    const char *c = (const char *)p;
    if (g_last_mirror >= 0 && g_last_mirror < (int)g_mirrors.size()) {
        const Mirror &m = g_mirrors[g_last_mirror];
        if (m.alive && c >= m.host && c < m.host + m.size) return g_last_mirror;
    }
    for (int i = 0; i < (int)g_mirrors.size(); i++) {
        const Mirror &m = g_mirrors[i];
        if (m.alive && c >= m.host && c < m.host + m.size) return g_last_mirror = i;
    }
    return -1;
}

Mirror &mirror_alloc(Mirror &m) {
    if (!m.dev) {
        ensure_backend();
        m.dev = (char *)fl_dev_malloc(m.size);
        if (!m.dev) B200_FAIL("device mirror of %zu bytes: %s", m.size, fl_last_error());
        if (g_verbose) fprintf(stderr, "[ggml_b200] mirror %p +%zu MiB -> dev %p%s\n", (const void *)m.host, m.size >> 20, (void *)m.dev, m.kind == MK_EXTERNAL ? " (external)" : m.kind == MK_SCRATCH ? " (scratch)" : "");
    }
    return m;
}
}  // namespace

static void packed_shards_clear();
static void drop_external_mirrors() {
    bool any = false;
    for (auto &m : g_mirrors)
        if (m.alive && m.kind == MK_EXTERNAL) { if (!any && fl_is_initialized()) fl_sync(); any = true; drop_mirror(m); m.alive = false; m.uploaded = 0; }
    if (any) packed_shards_clear();
    g_last_mirror = -1;
}
// Records of arenas that no open context covers any more.  Their buffers may have been freed, and foreign memory placed at those
// addresses later (a model file mapped where an earlier model's arena was) would otherwise resolve to the dead record: a stale
// device copy, or an upload that reads the old arena's length past the new memory.  Every arena in use re-registers at ggml_init.
static void drop_closed_arenas() {
    bool any = false;
    for (auto &m : g_mirrors) {
        if (!m.alive || m.kind != MK_ARENA) continue;
        bool open = false;
        for (const auto &slot : g_slots) open = open || (slot.used && slot.ctx.mem_buffer == m.host);
        if (open) continue;
        if (!any && fl_is_initialized()) fl_sync();
        any = true;
        drop_mirror(m);
        m.alive = false;
        m.uploaded = 0;
    }
    if (any) packed_shards_clear();
    g_last_mirror = -1;
}
static void mirrors_on_ctx_init(ggml_context *ctx) {
    // an arena re-created over the same buffer (Model::eval does this every call) re-uses its mirror
    int found = -1;
    for (int i = 0; i < (int)g_mirrors.size(); i++) {
        Mirror &m = g_mirrors[i];
        if (!m.alive) continue;
        const bool same = m.host == ctx->mem_buffer && m.size == ctx->mem_size;
        const bool overlap = m.host < ctx->mem_buffer + ctx->mem_size && ctx->mem_buffer < m.host + m.size;
        if (same) { found = i; if (m.uploaded) packed_shards_clear(); m.alloc_end = 0; m.uploaded = 0; m.kind = MK_ARENA; }
        else if (overlap) { drop_mirror(m); m.alive = false; }      // the buffer was re-allocated
    }
    if (found < 0) {
        g_mirrors.push_back(Mirror{ctx->mem_buffer, ctx->mem_size, nullptr, 0, 0, MK_ARENA, true});
        found = (int)g_mirrors.size() - 1;
    }
    ctx->mirror_id = found;
    g_last_mirror = -1;
    // A no_alloc context is how the reference loads a model whose tensors point into an mmap'ed file
    // (include/tensor/mem_context.hpp:12-16, lib/llama.cpp:213-258).  MK_EXTERNAL mirrors are keyed by host address only, and a
    // new mapping may land on the addresses of an earlier model's: everything registered for earlier mappings is stale now.
    // (A model that is still alive simply re-registers and re-uploads its tensors on next use.)
    if (ctx->no_alloc) {
        drop_external_mirrors();
        drop_closed_arenas();
    }
}
static void mirrors_on_ctx_free(ggml_context *) {}   // the arena (and its device mirror) outlives the context slot
static void mirrors_note_alloc(ggml_context *ctx, size_t end) {
    Mirror &m = g_mirrors[ctx->mirror_id];
    if (m.alive && m.host == ctx->mem_buffer && end > m.alloc_end) m.alloc_end = end;
}
static void mirrors_on_scratch(void *data, size_t size) {
    for (auto &m : g_mirrors)
        if (m.alive && m.host == (const char *)data && m.size == size) return;
    g_mirrors.push_back(Mirror{(const char *)data, size, nullptr, 0, 0, MK_SCRATCH, true});
}

// host pointer -> device pointer.  `compute_ctx` is the arena of the graph being run: nothing in it
// is uploaded here (its leafs are handled per graph).  Every other arena is persistent (weights, KV
// cache): whatever the allocator has handed out beyond the already-uploaded prefix is copied once;
// lower addresses are never re-copied, so data the device has written there (KV cache) is safe.
static char *dev_ptr(const void *host, size_t nbytes, const ggml_context *compute_ctx) {
    int i = find_mirror(host);
    if (i < 0) {
        // not inside any ggml arena: the tensor's data points at foreign memory (mmap'ed weights)
        g_mirrors.push_back(Mirror{(const char *)host, nbytes, nullptr, 0, 0, MK_EXTERNAL, true});
        i = (int)g_mirrors.size() - 1;
    }
    Mirror &m = mirror_alloc(g_mirrors[i]);
    const size_t off = (const char *)host - m.host;
    if (m.kind != MK_ARENA && off + nbytes > m.size)
        B200_FAIL("tensor at %p (+%zu) straddles the end of a registered range %p (+%zu)", host, nbytes, (const void *)m.host, m.size);
    size_t want = 0;
    if (m.kind == MK_EXTERNAL) want = m.size;
    else if (m.kind == MK_ARENA && !(compute_ctx && m.host == compute_ctx->mem_buffer)) want = std::min(m.size, m.alloc_end);
    if (want > m.uploaded) {
        if (g_verbose) fprintf(stderr, "[ggml_b200] upload %p [%zu, %zu) -> device\n", (const void *)m.host, m.uploaded, want);
        FLC(fl_h2d(m.dev + m.uploaded, m.host + m.uploaded, want - m.uploaded));
        m.uploaded = want;
    }
    return m.dev + off;
}

static void tp_gather_kv();
// a device op is about to write `host`'s mirror: remember it if the arena is persistent (the KV cache)
static void mark_device_write(const void *host, const ggml_context *compute_ctx) {
    const int i = find_mirror(host);
    if (i < 0) return;
    Mirror &m = g_mirrors[i];
    if (m.kind == MK_ARENA && !(compute_ctx && m.host == compute_ctx->mem_buffer) && !m.device_dirty) { m.device_dirty = true; g_dirty_arenas.fetch_add(1, std::memory_order_release); }
}
// The reference reads and overwrites kv_self.{k,v}->data on the host in KVCacheBuffer::save_state / load_state
// (reference lib/llama.cpp:57-78) with no ggml call in between -- except ggml_nbytes(k), evaluated as an argument right
// before each access.  So the exported ggml_nbytes is the hook that keeps the unchanged bridge correct: when it is called
// on a tensor of a persistent arena the device has written, the arena is copied back to the host (save_state then sees
// current data) and marked for re-upload before the next graph (load_state's data then reaches the device).  It never
// fires during eval: Model::eval does not call ggml_nbytes on KV tensors, and the flag is clear outside device writes.
static void host_access_hook(const struct ggml_tensor *t) {
    static const bool off = getenv("FASTLLAMA_B200_NO_HOST_HOOK") != nullptr;      // debugging aid: show what breaks without it
    static std::mutex hook_mutex;                                                  // the slow path mutates the mirror table
    std::lock_guard<std::mutex> lock(hook_mutex);
    if (off || !t || !t->data || g_mirrors.empty()) return;
    const int i = find_mirror(t->data);
    if (i < 0) return;
    Mirror &m = g_mirrors[i];
    if (!m.device_dirty || !m.dev) return;
    if (fl_comm_world() > 1 && g_tp_kv_sharded) tp_gather_kv();      // collective: every rank saves / loads its state at the same point
    const size_t n = std::min(m.uploaded, std::min(m.size, m.alloc_end));
    if (g_verbose) fprintf(stderr, "[ggml_b200] host access to device-written arena %p: syncing %zu MiB back, re-upload before the next graph\n", (const void *)m.host, n >> 20);
    FLC(fl_sync());
    if (n) FLC(fl_d2h((void *)m.host, m.dev, n));
    FLC(fl_sync());
    m.device_dirty = false;
    g_dirty_arenas.fetch_sub(1, std::memory_order_release);
    m.uploaded = 0;              // the host may now change the data (load_state): everything is uploaded again on next use
}

extern "C" void ggml_b200_invalidate(const void *ptr, size_t size) {
    const int i = find_mirror(ptr);
    if (i < 0 || !g_mirrors[i].dev) return;
    Mirror &m = g_mirrors[i];
    const size_t off = (const char *)ptr - m.host;
    const size_t end = std::min(off + size, m.uploaded);
    if (end > off) FLC(fl_h2d(m.dev + off, m.host + off, end - off));
}
extern "C" void ggml_b200_sync_to_host(const void *ptr, size_t size) {
    const int i = find_mirror(ptr);
    if (i < 0 || !g_mirrors[i].dev) return;
    Mirror &m = g_mirrors[i];
    const size_t off = (const char *)ptr - m.host;
    const size_t n = std::min(size, m.size - off);
    FLC(fl_d2h((void *)(m.host + off), m.dev + off, n));
    FLC(fl_sync());
}
static void decode_state_release();
// Frees every device resource of the backend: decode graph / token plan / workspace, tensor-parallel shards, all mirrors.
// fastllama_b200.Model.close() calls it after llama_free_context; the next model starts from a clean device.
extern "C" void ggml_b200_release_all(void) {
    if (fl_is_initialized()) fl_sync();
    decode_state_release();
    packed_shards_clear();
    for (auto &m : g_mirrors) {
        drop_mirror(m);
        m.uploaded = 0;
        if (m.device_dirty) { m.device_dirty = false; g_dirty_arenas.fetch_sub(1, std::memory_order_release); }
        if (m.kind != MK_ARENA) m.alive = false;
    }
    // an arena whose context is still open keeps its record (lookups are by address); the others are forgotten
    drop_closed_arenas();
}
// how the last single-token eval ran: 0 = node-by-node executor, 1 = fused plan with one kernel per matrix group,
// 2 = fused plan as one persistent kernel per token (fl_token_kernel.cu)
extern "C" int ggml_b200_decode_mode(void) { return g_decode_mode; }
extern "C" void ggml_b200_get_host_profile(double out[8], int reset) {
    for (int i = 0; i < 8; i++) { out[i] = g_hostprof[i]; if (reset) g_hostprof[i] = 0; }
}
extern "C" void ggml_b200_set_profile(int on) {
    ensure_backend();
    if (!g_pev0) { g_pev0 = fl_event_create(); g_pev1 = fl_event_create(); }
    g_profile = on != 0;
    if (on) g_kstats.clear();
}
extern "C" int ggml_b200_get_kernel_stats(struct ggml_b200_kernel_stat *out, int max_entries) {
    const int n = std::min((int)g_kstats.size(), max_entries);
    for (int i = 0; i < n; i++) out[i] = g_kstats[i];
    return n;
}
extern "C" void ggml_b200_get_stats(struct ggml_b200_stats *out) {
    out->n_evals = g_stats.n_evals;
    out->last_eval_device_us = g_stats.last_us;
    out->total_device_us = g_stats.total_us;
    out->launches = fl_is_initialized() ? fl_launch_count() : 0;
    out->graph_replays = g_stats.graph_replays;
}

// ================================================================================================
// 3. executor
// ================================================================================================
namespace {
struct Exec {
    const ggml_context *ctx;
    void *q8_work = nullptr;     // device scratch for quantised activations (the reference's "wdata")
    size_t q8_cap = 0;
};
Exec g_exec;

fl_view view_of(const ggml_tensor *t, const ggml_context *cctx) {
    fl_view v;
    v.data = dev_ptr(t->data, nbytes_of(t), cctx);
    for (int i = 0; i < 4; i++) { v.ne[i] = t->ne[i]; v.nb[i] = (int64_t)t->nb[i]; }
    return v;
}

void need_f32(const ggml_tensor *t, const char *what) {
    if (t->type != GGML_TYPE_F32) B200_FAIL("%s: tensor type %s is not supported by the B200 backend (f32 only)", what, k_tname[t->type]);
}

void exec_mul_mat(const ggml_tensor *node, const ggml_context *cctx) {
    const ggml_tensor *a = node->src0, *b = node->src1;
    need_f32(b, "mul_mat src1");
    if (a->type == GGML_TYPE_F32 && a->ne[2] == 1 && a->ne[3] == 1 && b->ne[2] == 1 && b->ne[3] == 1 && a->ne[0] <= 256 && a->nb[0] == 4 && b->nb[0] == 4 &&
        node->nb[0] == 4) {
        // two plain f32 matrices with a short contraction (B*A of a LoRA adapter, reference lib/llama.cpp:867): the reference's exact
        // summation order, so that the merged weights re-quantise to the reference's bytes
        FLC(fl_dev_mul_mat_f32_ref((const float *)dev_ptr(a->data, nbytes_of(a), cctx), a->nb[1] / 4, (int)a->ne[1], (const float *)dev_ptr(b->data, nbytes_of(b), cctx),
                                   b->nb[1] / 4, (int)b->ne[1], (int)a->ne[0], (float *)dev_ptr(node->data, nbytes_of(node), cctx), node->nb[1] / 4));
        return;
    }
    if (a->type == GGML_TYPE_F32) {
        fl_view va = view_of(a, cctx), vb = view_of(b, cctx), vd = view_of(node, cctx);
        FLC(fl_dev_mul_mat_f32(&va, &vb, &vd));
        return;
    }
    if (a->type != GGML_TYPE_Q4_0 && a->type != GGML_TYPE_Q4_1)
        B200_FAIL("mul_mat: weight type %s is not supported by the B200 backend (q4_0, q4_1, f32)", k_tname[a->type]);
    // ggml_compute_forward_mul_mat_q_f32 preconditions (reference lib/ggml.c:7969-7991)
    B200_ASSERT(a->ne[2] == 1 && a->ne[3] == 1 && b->ne[2] == 1 && b->ne[3] == 1);
    B200_ASSERT(a->nb[0] == k_tsize[a->type] && b->nb[0] == sizeof(float) && node->nb[0] == sizeof(float));
    B200_ASSERT(a->ne[0] % 32 == 0 && a->ne[0] == b->ne[0]);
    const int M = (int)a->ne[1], K = (int)a->ne[0], N = (int)b->ne[1];
    const size_t q8_bytes = (size_t)(K / 32) * 40 * (size_t)N;
    if (g_exec.q8_cap < q8_bytes) {
        if (g_exec.q8_work) FLC(fl_dev_free(g_exec.q8_work));
        g_exec.q8_cap = std::max(q8_bytes, (size_t)1 << 20);
        g_exec.q8_work = fl_dev_malloc(g_exec.q8_cap);
        if (!g_exec.q8_work) B200_FAIL("q8_0 work buffer: %s", fl_last_error());
    }
    const char *W = dev_ptr(a->data, nbytes_of(a), cctx);
    const float *X = (const float *)dev_ptr(b->data, nbytes_of(b), cctx);
    float *D = (float *)dev_ptr(node->data, nbytes_of(node), cctx);
    // INIT phase: src1 rows -> q8_0 (reference lib/ggml.c:8105-8119)
    FLC(fl_dev_quantize_q8_0(X, b->nb[1], g_exec.q8_work, K, N));
    // COMPUTE phase (reference lib/ggml.c:8125-8163)
    if (g_profile) FLC(fl_event_record(g_pev0));
    FLC(fl_dev_mul_mat_q((int)a->type, W, a->nb[1], M, K, g_exec.q8_work, N, D, node->nb[1] / sizeof(float), 0));
    if (g_profile) {
        FLC(fl_event_record(g_pev1));
        FLC(fl_event_sync(g_pev1));
        float ms = 0.f;
        FLC(fl_event_elapsed_ms(g_pev0, g_pev1, &ms));
        ggml_b200_kernel_stat *e = nullptr;
        for (auto &k : g_kstats) if (k.type == (int)a->type && k.M == M && k.K == K && k.N == N) e = &k;
        if (!e) {
            g_kstats.push_back(ggml_b200_kernel_stat{(int)a->type, M, K, N, 0, 0.0,
                                                     (double)M * (K / 32) * (double)k_tsize[a->type] + (double)(K / 32) * 40.0 * N + 4.0 * M * N});
            e = &g_kstats.back();
        }
        e->launches++;
        e->total_ms += ms;
    }
}

void exec_node(ggml_tensor *node, const ggml_context *cctx) {
    switch (node->op) {
        case GGML_OP_NONE: case GGML_OP_RESHAPE: case GGML_OP_VIEW: case GGML_OP_PERMUTE: case GGML_OP_TRANSPOSE:
            return;                                   // pure address arithmetic, already in node->data / nb
        default: break;
    }
    mark_device_write(node->data, cctx);              // a cpy into a KV-cache view lands in a persistent arena
    switch (node->op) {
        case GGML_OP_GET_ROWS: {
            const ggml_tensor *a = node->src0, *ids = node->src1;
            if (a->type != GGML_TYPE_Q4_0 && a->type != GGML_TYPE_Q4_1)
                B200_FAIL("get_rows: table type %s is not supported by the B200 backend (q4_0, q4_1)", k_tname[a->type]);
            FLC(fl_dev_dequantize_rows((int)a->type, dev_ptr(a->data, nbytes_of(a), cctx), a->nb[1], (int)a->ne[0],
                                       (const int32_t *)dev_ptr(ids->data, nbytes_of(ids), cctx), (int)ggml_nelements(ids),
                                       (float *)dev_ptr(node->data, nbytes_of(node), cctx), node->nb[1] / sizeof(float)));
            return;
        }
        case GGML_OP_RMS_NORM: {
            need_f32(node->src0, "rms_norm");
            fl_view s = view_of(node->src0, cctx), d = view_of(node, cctx);
            FLC(fl_dev_rms_norm(&s, &d));
            return;
        }
        case GGML_OP_ADD: case GGML_OP_MUL: {
            if (node->op == GGML_OP_ADD && (node->src0->type == GGML_TYPE_Q4_0 || node->src0->type == GGML_TYPE_Q4_1)) {
                // W (+)= f32 matrix: the LoRA merge, ggml_compute_forward_add_q_f32 (reference lib/ggml.c:6414-6520)
                const ggml_tensor *a = node->src0, *b = node->src1;
                need_f32(b, "add (quantised + f32) src1");
                B200_ASSERT(node->type == a->type && same_shape(a, b) && same_shape(a, node) && a->ne[2] == 1 && a->ne[3] == 1);
                B200_ASSERT(a->nb[0] == k_tsize[a->type] && b->nb[0] == sizeof(float) && node->nb[0] == k_tsize[a->type] && a->ne[0] % 32 == 0);
                FLC(fl_dev_add_q_f32((int)a->type, dev_ptr(a->data, nbytes_of(a), cctx), a->nb[1], (int)a->ne[1], (int)a->ne[0],
                                     (const float *)dev_ptr(b->data, nbytes_of(b), cctx), b->nb[1] / sizeof(float), dev_ptr(node->data, nbytes_of(node), cctx), node->nb[1]));
                // the host tensor follows the device (tensor-parallel shards are uploaded from the HOST tensor, and a mirror that is
                // dropped later would otherwise come back with the unmerged bytes)
                FLC(fl_d2h(node->data, dev_ptr(node->data, nbytes_of(node), cctx), nbytes_of(node)));
                FLC(fl_sync());
                packed_shards_clear();          // shards cut from the old weights are stale now
                return;
            }
            need_f32(node->src0, k_opname[node->op]); need_f32(node->src1, k_opname[node->op]);
            fl_view a = view_of(node->src0, cctx), b = view_of(node->src1, cctx), d = view_of(node, cctx);
            if (node->op == GGML_OP_ADD) FLC(fl_dev_add(&a, &b, &d)); else FLC(fl_dev_mul(&a, &b, &d));
            return;
        }
        case GGML_OP_REPEAT: {
            need_f32(node->src0, "repeat");
            fl_view s = view_of(node->src0, cctx), d = view_of(node, cctx);
            FLC(fl_dev_repeat(&s, &d));
            return;
        }
        case GGML_OP_SILU: {
            need_f32(node->src0, "silu");
            fl_view s = view_of(node->src0, cctx), d = view_of(node, cctx);
            FLC(fl_dev_silu(&s, &d));
            return;
        }
        case GGML_OP_MUL_MAT:
            exec_mul_mat(node, cctx);
            return;
        case GGML_OP_SCALE: {
            need_f32(node->src0, "scale");
            if (node->src1->op != GGML_OP_NONE) B200_FAIL("scale: the factor must be a host constant (ggml_new_f32)");
            fl_view d = view_of(node, cctx);
            FLC(fl_dev_scale(&d, *(const float *)node->src1->data));
            return;
        }
        case GGML_OP_DIAG_MASK_INF: {
            need_f32(node->src0, "diag_mask_inf");
            fl_view d = view_of(node, cctx);
            FLC(fl_dev_diag_mask_inf(&d, *(const int32_t *)node->src1->data));
            return;
        }
        case GGML_OP_SOFT_MAX: {
            need_f32(node->src0, "soft_max");
            fl_view d = view_of(node, cctx);
            FLC(fl_dev_soft_max(&d));
            return;
        }
        case GGML_OP_ROPE: {
            need_f32(node->src0, "rope");
            const int32_t *p = (const int32_t *)node->src1->data;
            fl_view d = view_of(node, cctx);
            FLC(fl_dev_rope(&d, p[0], p[1], p[2]));
            return;
        }
        case GGML_OP_CPY: case GGML_OP_DUP: case GGML_OP_CONT: {
            need_f32(node->src0, "cpy src"); need_f32(node, "cpy dst (an f16 KV cache is not supported)");
            fl_view s = view_of(node->src0, cctx), d = view_of(node, cctx);
            FLC(fl_dev_cpy_f32(&s, &d));
            return;
        }
        default:
            B200_FAIL("op %s is outside the LLaMA eval set and has no B200 implementation (and there is no CPU fallback)", k_opname[node->op]);
    }
}

inline bool in_ctx(const ggml_context *c, const void *p) {
    return c && (const char *)p >= c->mem_buffer && (const char *)p < c->mem_buffer + c->mem_size;
}

// ================================================================================================
// 3b. the fused decode plan
//
// Model::eval with one token always emits the same 37-node layer (reference lib/llama.cpp:310-455;
// node order = depth-first post-order of ggml_build_forward_expand).  When a graph matches that
// template exactly it is lowered to 5 kernels per layer (fl_cuda.h "fused decode step") and the
// whole token step is captured once into a CUDA graph that is replayed for every later token: all
// device addresses are the same from token to token (the compute arena is re-built identically), only
// n_past and the token id change, and both are read from device memory.  Anything that does not
// match falls through to the node-by-node executor (still on the GPU).
// ================================================================================================
struct LayerPlan {
    fl_mv_args qkv, wo, w13, w2;
    const float *q, *kcache, *vcache;
    float *att;
};
struct DecodePlan {
    int n_layer = 0, n_embd = 0, n_head = 0, n_ctx = 0, n_past = 0;
    float scale = 0.f;
    // embedding gather
    int emb_type = 0, emb_K = 0;
    const void *emb_w = nullptr;
    size_t emb_stride = 0;
    const int32_t *emb_ids = nullptr;
    float *emb_dst = nullptr;
    std::vector<LayerPlan> layers;
    fl_mv_args head;
    int world = 1, heads_local = 0;             // tensor-parallel degree and heads per rank
    float *logits_local = nullptr, *logits_all = nullptr;
    int vocab_local = 0;
};
// Private device workspace of the decode step.  The compute arena cannot be used for intermediates:
// its layout shifts from token to token (the K*Q score tensor grows with n_past), and the captured
// graph needs addresses that never move.
struct DecodeWs {
    int n_embd = 0, n_ff = 0, n_vocab = 0;
    float *xa = nullptr, *xb = nullptr, *q = nullptr, *att = nullptr, *ff = nullptr, *m1 = nullptr, *m3 = nullptr, *emb = nullptr, *logits = nullptr;
    float *logits_local = nullptr;
    int32_t *d_tok = nullptr;
    // The dataflow ("LL") vectors of the token kernel (include/fl_cuda.h, fl_mv_args): {value, epoch} words that hand the
    // activations from step to step without grid barriers.  Layout of the buffer: 4096 bytes of counters (word 0 = the running epoch),
    // then X (the residual stream, n_embd words), A (attention output), B (x + wo.att) and H (the FFN's hidden vector, n_ff words).
    // One GPU: plain device memory.  Tensor parallel: the buffer of fl_comm_shared_alloc, peers[r] = rank r's buffer as mapped here;
    // every rank stores its row slice of a vector into ALL buffers (NVLink), so each holds the complete gathered vector.
    void *ll_local = nullptr;   // world == 1: owned here
    void *peers[8] = {nullptr};
    bool peer_mapped = false;
    size_t ll_cap_embd = 0, ll_cap_ff = 0;      // the element counts the buffer was laid out for
};
struct DecodeState {
    DecodePlan plan;            // the plan the captured graph was built from
    DecodeWs ws;
    void *graph = nullptr;
    void *token_plan = nullptr;   // the persistent per-token kernel's program (single-GPU decode)
    int *d_npast = nullptr;
    int *h_scalars = nullptr;   // pinned: [0] n_past, [1] token id
    char *h_out = nullptr;      // pinned staging of the step's results (logits, then the embeddings row): the caller's arena is pageable
    size_t h_out_cap = 0;
    bool enabled = true, use_graph = true, use_token_kernel = true, inited = false;
    bool no_token_plan = false;       // the current plan's graph is not one the token kernel takes: node-by-node execution
    bool tp_kv_sharded = false;   // tensor-parallel decode steps have written only this rank's heads into the KV cache ...
    int tp_first_pos = 0, tp_end_pos = 0;   // ... for positions [tp_first_pos, tp_end_pos)
};
struct DecodeOutputs { const void *kv_host = nullptr; void *logits_host = nullptr; size_t logits_bytes = 0; void *emb_host = nullptr; size_t emb_bytes = 0; int32_t token = 0; };
DecodeState g_dec;

struct Cur {
    ggml_cgraph *g;
    int i;
    bool ok;
    ggml_tensor *next(ggml_op op) {
        if (!ok || i >= g->n_nodes || g->nodes[i]->op != op) { ok = false; return nullptr; }
        return g->nodes[i++];
    }
};
#define PM(cond) do { if (!(cond)) { if (g_verbose) fprintf(stderr, "[ggml_b200] decode plan: no match (line %d): %s\n", __LINE__, #cond); return false; } } while (0)

inline bool is_qw(const ggml_tensor *w) {
    return w && w->op == GGML_OP_NONE && (w->type == GGML_TYPE_Q4_0 || w->type == GGML_TYPE_Q4_1) && w->ne[2] == 1 && w->ne[3] == 1 &&
           w->nb[0] == k_tsize[w->type] && w->nb[1] == (size_t)(w->ne[0] / 32) * k_tsize[w->type];
}
inline bool is_vec(const ggml_tensor *t, int64_t n) {
    return t && t->type == GGML_TYPE_F32 && t->ne[0] == n && t->ne[1] == 1 && t->ne[2] == 1 && t->ne[3] == 1 && t->nb[0] == 4;
}
template <typename T> inline T *dp(const ggml_tensor *t, const ggml_context *c) { return (T *)dev_ptr(t->data, nbytes_of(t), c); }

void mv_base(fl_mv_args &a, int type, int K) {
    memset(&a, 0, sizeof(a));
    a.type = type;
    a.K = K;
}

void ensure_ws(DecodeWs &w, int n_embd, int n_ff, int n_vocab) {
    if (w.xa && w.n_embd == n_embd && w.n_ff == n_ff && w.n_vocab == n_vocab) return;
    if (w.xa) { FLC(fl_sync()); FLC(fl_dev_free(w.xa)); }
    const size_t total = (size_t)n_embd * 6 + (size_t)n_ff * 2 + (size_t)n_vocab * 2 + 64;
    float *base = (float *)fl_dev_malloc(total * sizeof(float));
    if (!base) B200_FAIL("decode workspace: %s", fl_last_error());
    w.xa = base; w.xb = w.xa + n_embd; w.q = w.xb + n_embd; w.att = w.q + n_embd; w.ff = w.att + n_embd; w.emb = w.ff + n_embd;
    w.m1 = w.emb + n_embd; w.m3 = w.m1 + n_ff; w.logits = w.m3 + n_ff; w.logits_local = w.logits + n_vocab;
    w.d_tok = (int32_t *)(w.logits_local + n_vocab);
    w.n_embd = n_embd; w.n_ff = n_ff; w.n_vocab = n_vocab;
    const int world = fl_comm_world(), rank = fl_comm_rank();
    if (world > 1) {
        // collective: every rank gets here on its first decode step.  The peer-mapped buffer is per process (it cannot be freed), so it
        // is laid out for the largest model of the family (n_embd 8192, n_ff 22016) or this one, whichever is larger.
        if (!w.peer_mapped) {
            w.ll_cap_embd = (size_t)std::max(n_embd, 8192); w.ll_cap_ff = (size_t)std::max(n_ff, 22016);
            if (fl_comm_shared_alloc(4096 + (3 * w.ll_cap_embd + w.ll_cap_ff) * 8, w.peers) != 0)
                B200_FAIL("tensor-parallel decode needs peer-mapped buffers between the GPUs: %s", fl_last_error());
            w.peer_mapped = true;
        }
        if ((size_t)n_embd > w.ll_cap_embd || (size_t)n_ff > w.ll_cap_ff) B200_FAIL("tensor-parallel decode: model wider than the peer-mapped vectors (n_embd %d, n_ff %d)", n_embd, n_ff);
    } else {
        if (w.ll_local && ((size_t)n_embd > w.ll_cap_embd || (size_t)n_ff > w.ll_cap_ff)) { FLC(fl_sync()); FLC(fl_dev_free(w.ll_local)); w.ll_local = nullptr; }
        if (!w.ll_local) {
            w.ll_cap_embd = (size_t)n_embd; w.ll_cap_ff = (size_t)n_ff;
            const size_t bytes = 4096 + (3 * w.ll_cap_embd + w.ll_cap_ff) * 8;
            w.ll_local = fl_dev_malloc(bytes);
            if (!w.ll_local) B200_FAIL("decode workspace: %s", fl_last_error());
            FLC(fl_dev_memset(w.ll_local, 0, bytes));              // epoch 0 is never expected: nothing has arrived yet
        }
        w.peers[0] = w.ll_local;
    }
    (void)rank;
}

// ---- tensor-parallel weight shards, uploaded straight from the HOST tensors (reference hook point lib/llama.cpp:257-258) -----------
// Under tensor parallelism a rank never uploads the model: every weight the fused decode plan touches gets a private device copy of
// exactly what this rank reads -- a row range (wq/wk/wv/w1/w3/output: contiguous host bytes), a K-slice (wo/w2: blocks
// [blk0, blk0 + nblk) of every row, gathered on the host into pinned staging so that the device never sees the other ranks' columns;
// the packed row stride is a 16-byte multiple so every tile is still one bulk copy), or the whole tensor (norm weights, the
// embedding table).  8 ranks of a 65B model upload 5 GB each instead of 40.6 GB.  The arena / mmap mirrors of the weights are not
// touched by decode steps at all; a replicated multi-token eval (n_batch > 1) still mirrors what it reads.
struct ShardKey {
    const void *host; int kind, a, b;
    bool operator==(const ShardKey &o) const { return host == o.host && kind == o.kind && a == o.a && b == o.b; }
};
struct ShardKeyHash { size_t operator()(const ShardKey &k) const { return std::hash<const void *>()(k.host) ^ ((size_t)k.kind * 0x9E3779B97F4A7C15ull) ^ ((size_t)k.a << 20) ^ (size_t)k.b; } };
enum { SH_FULL = 0, SH_ROWS = 1, SH_COLS = 2 };
std::unordered_map<ShardKey, void *, ShardKeyHash> g_packed;
char *g_shard_staging = nullptr;
size_t g_shard_staging_cap = 0, g_shard_bytes = 0;
}  // namespace
static void packed_shards_clear() {
    if (g_packed.empty()) return;
    if (fl_is_initialized()) fl_sync();
    for (auto &kv : g_packed) fl_dev_free(kv.second);
    g_packed.clear();
    g_shard_bytes = 0;
}
namespace {
// device copy of (kind SH_FULL) the whole tensor, (SH_ROWS) rows [a, a + b), (SH_COLS) blocks [a, a + b) of every row with row stride *stride_out
const void *tp_shard(const ggml_tensor *w, int kind, int a, int b, size_t *stride_out = nullptr) {
    const size_t bb = k_tsize[w->type];
    const size_t stride = kind == SH_COLS ? (((size_t)b * bb + 15) & ~(size_t)15) : w->nb[1];
    if (stride_out) *stride_out = stride;
    const ShardKey key{w->data, kind, a, b};
    auto it = g_packed.find(key);
    if (it != g_packed.end()) return it->second;
    ensure_backend();
    const size_t rows = (size_t)nrows(w);
    const size_t bytes = kind == SH_FULL ? nbytes_of(w) : kind == SH_ROWS ? (size_t)b * w->nb[1] : stride * rows;
    void *dst = fl_dev_malloc(bytes + 256);
    if (!dst) B200_FAIL("tensor-parallel shard of %zu bytes: %s", bytes, fl_last_error());
    if (kind == SH_COLS) {
        // gather the K-slice on the host: the other ranks' columns never cross PCIe
        if (g_shard_staging_cap < bytes) {
            if (g_shard_staging) { FLC(fl_sync()); FLC(fl_host_free_pinned(g_shard_staging)); }
            g_shard_staging_cap = bytes + bytes / 4;
            g_shard_staging = (char *)fl_host_alloc_pinned(g_shard_staging_cap);
            if (!g_shard_staging) B200_FAIL("shard staging: %s", fl_last_error());
        }
        FLC(fl_sync());                                               // the previous shard has left the staging buffer
        const size_t slice = (size_t)b * bb;
        for (size_t r = 0; r < rows; r++) {
            char *d = g_shard_staging + r * stride;
            memcpy(d, (const char *)w->data + r * w->nb[1] + (size_t)a * bb, slice);
            if (stride > slice) memset(d + slice, 0, stride - slice);
        }
        FLC(fl_h2d(dst, g_shard_staging, bytes));
    } else {
        FLC(fl_h2d(dst, (const char *)w->data + (kind == SH_ROWS ? (size_t)a * w->nb[1] : 0), bytes));
    }
    g_packed[key] = dst;
    g_shard_bytes += bytes;
    if (g_verbose && (g_packed.size() & 63) == 0) fprintf(stderr, "[ggml_b200] tensor-parallel shards: %zu tensors, %zu MiB on the device\n", g_packed.size(), g_shard_bytes >> 20);
    return dst;
}

bool match_decode(const ggml_context *ctx, ggml_cgraph *g, DecodePlan &P, DecodeWs &W, DecodeOutputs &O) {
    const int world = fl_comm_world(), rank = fl_comm_rank();
    // weights: one GPU -> the arena / mmap mirror; tensor parallel -> only this rank's shard, uploaded from the host tensor (tp_shard)
    auto wfull = [&](const ggml_tensor *t) -> const void * { return world == 1 ? (const void *)dp<const void>(t, ctx) : tp_shard(t, SH_FULL, 0, 0); };
    auto wrows = [&](const ggml_tensor *t, int row0, int n) -> const void * {
        return world == 1 ? (const void *)((const char *)dp<const void>(t, ctx) + (size_t)row0 * t->nb[1]) : tp_shard(t, SH_ROWS, row0, n);
    };
    PM(g->n_nodes >= 4 + 37 && (g->n_nodes - 4) % 37 == 0);
    Cur c{g, 0, true};
    ggml_tensor *n0 = c.next(GGML_OP_GET_ROWS);
    PM(n0 && is_qw(n0->src0) && n0->src1 && n0->src1->type == GGML_TYPE_I32 && ggml_nelements(n0->src1) == 1);
    const int n_embd = (int)n0->src0->ne[0];
    PM(is_vec(n0, n_embd));
    P.n_embd = n_embd;
    P.n_layer = (g->n_nodes - 4) / 37;
    P.emb_type = (int)n0->src0->type; P.emb_K = n_embd; P.emb_stride = n0->src0->nb[1];
    P.emb_w = wfull(n0->src0);
    O.token = *(const int32_t *)n0->src1->data;
    P.layers.resize(P.n_layer);
    ggml_tensor *x = n0;
    int n_past = -1, n_head = -1, n_ctx = -1;
    float *xin = nullptr, *xout = nullptr;     // residual stream ping-pong in the workspace
    for (int il = 0; il < P.n_layer; il++) {
        LayerPlan &L = P.layers[il];
        ggml_tensor *a = c.next(GGML_OP_RMS_NORM), *b = c.next(GGML_OP_MUL);
        PM(c.ok && a->src0 == x && b->src1 == a && is_vec(b->src0, n_embd) && b->src0->op == GGML_OP_NONE);
        // K
        ggml_tensor *mk = c.next(GGML_OP_MUL_MAT), *rsk = c.next(GGML_OP_RESHAPE), *rk = c.next(GGML_OP_ROPE), *vk = c.next(GGML_OP_VIEW),
                    *ck = c.next(GGML_OP_CPY);
        PM(c.ok && is_qw(mk->src0) && mk->src1 == b && rsk->src0 == mk && rk->src0 == rsk && ck->src0 == rk && ck->src1 == vk);
        const int hd = (int)rsk->ne[0];
        PM(hd > 0 && n_embd % hd == 0 && rsk->ne[1] == n_embd / hd && rsk->ne[2] == 1);
        const int32_t *rp = (const int32_t *)rk->src1->data;
        PM(rp[1] == hd && rp[2] == 0 && hd % 2 == 0);
        if (il == 0) { n_past = rp[0]; n_head = n_embd / hd; }
        PM(rp[0] == n_past && vk->type == GGML_TYPE_F32 && vk->src0 && vk->src0->op == GGML_OP_NONE);
        // V
        ggml_tensor *mvv = c.next(GGML_OP_MUL_MAT), *rsv = c.next(GGML_OP_RESHAPE), *tv = c.next(GGML_OP_TRANSPOSE), *vv = c.next(GGML_OP_VIEW),
                    *cv = c.next(GGML_OP_CPY);
        PM(c.ok && is_qw(mvv->src0) && mvv->src1 == b && rsv->src0 == mvv && tv->src0 == rsv && cv->src0 == tv && cv->src1 == vv);
        PM(vv->type == GGML_TYPE_F32 && vv->ne[0] == 1 && vv->ne[1] == n_embd && vv->nb[1] % 4 == 0);
        const int nctx_l = (int)(vv->nb[1] / 4);
        if (il == 0) n_ctx = nctx_l;
        PM(nctx_l == n_ctx && n_past < n_ctx);
        // cache views used by attention
        ggml_tensor *Vv = c.next(GGML_OP_VIEW), *Kv = c.next(GGML_OP_VIEW), *Kr = c.next(GGML_OP_RESHAPE), *Kp = c.next(GGML_OP_PERMUTE);
        PM(c.ok && Kr->src0 == Kv && Kp->src0 == Kr && Vv->src0 == vv->src0 && Kv->src0 == vk->src0);
        PM(Kv->ne[0] == (int64_t)(n_past + 1) * n_embd && Vv->ne[0] == n_past + 1 && Vv->ne[1] == hd && Vv->ne[2] == n_head &&
           Vv->nb[1] == (size_t)n_ctx * 4 && Vv->nb[2] == (size_t)n_ctx * 4 * hd);
        // the slots written this step must be position n_past of this layer's cache
        PM((char *)vk->data == (char *)Kv->data + (size_t)n_past * n_embd * 4 && (char *)vv->data == (char *)Vv->data + (size_t)n_past * 4);
        // Q
        ggml_tensor *mq = c.next(GGML_OP_MUL_MAT), *rsq = c.next(GGML_OP_RESHAPE), *rq = c.next(GGML_OP_ROPE), *pq = c.next(GGML_OP_PERMUTE);
        PM(c.ok && is_qw(mq->src0) && mq->src1 == b && rsq->src0 == mq && rq->src0 == rsq && pq->src0 == rq);
        const int32_t *rpq = (const int32_t *)rq->src1->data;
        PM(rpq[0] == n_past && rpq[1] == hd && rpq[2] == 0);
        // attention
        ggml_tensor *kq = c.next(GGML_OP_MUL_MAT), *sc = c.next(GGML_OP_SCALE), *mask = c.next(GGML_OP_DIAG_MASK_INF), *sm = c.next(GGML_OP_SOFT_MAX),
                    *kqv = c.next(GGML_OP_MUL_MAT), *pm = c.next(GGML_OP_PERMUTE), *att = c.next(GGML_OP_CPY);
        PM(c.ok && kq->src0 == Kp && kq->src1 == pq && sc->src0 == kq && mask->src0 == sc && sm->src0 == mask && kqv->src0 == Vv && kqv->src1 == sm &&
           pm->src0 == kqv && att->src0 == pm && is_vec(att, n_embd) && ggml_nelements(sc->src1) == 1 && sc->src1->op == GGML_OP_NONE);
        PM(*(const int32_t *)mask->src1->data == n_past);
        const float scale = *(const float *)sc->src1->data;
        if (il == 0) P.scale = scale;
        PM(scale == P.scale);
        // output projection + residual
        ggml_tensor *mo = c.next(GGML_OP_MUL_MAT), *ff = c.next(GGML_OP_ADD);
        PM(c.ok && is_qw(mo->src0) && mo->src1 == att && ff->src0 == mo && ff->src1 == x);
        // feed-forward
        ggml_tensor *cn = c.next(GGML_OP_RMS_NORM), *d = c.next(GGML_OP_MUL), *m1 = c.next(GGML_OP_MUL_MAT), *s1 = c.next(GGML_OP_SILU),
                    *m3 = c.next(GGML_OP_MUL_MAT), *h = c.next(GGML_OP_MUL), *m2 = c.next(GGML_OP_MUL_MAT), *xo = c.next(GGML_OP_ADD);
        PM(c.ok && cn->src0 == ff && d->src1 == cn && is_vec(d->src0, n_embd) && d->src0->op == GGML_OP_NONE && is_qw(m1->src0) && m1->src1 == d &&
           s1->src0 == m1 && is_qw(m3->src0) && m3->src1 == d && h->src0 == s1 && h->src1 == m3 && is_qw(m2->src0) && m2->src1 == h &&
           xo->src0 == m2 && xo->src1 == ff);
        const ggml_tensor *wq = mq->src0, *wk = mk->src0, *wv = mvv->src0, *wo = mo->src0, *w1 = m1->src0, *w3 = m3->src0, *w2 = m2->src0;
        const int n_ff = (int)w1->ne[1];
        PM(wq->type == wk->type && wq->type == wv->type && w1->type == w3->type);
        PM(wq->ne[0] == n_embd && wk->ne[0] == n_embd && wv->ne[0] == n_embd && wq->ne[1] == n_embd && wk->ne[1] == n_embd && wv->ne[1] == n_embd);
        PM(wo->ne[0] == n_embd && wo->ne[1] == n_embd && w1->ne[0] == n_embd && w3->ne[0] == n_embd && w3->ne[1] == n_ff && w2->ne[0] == n_ff &&
           w2->ne[1] == n_embd);
        PM(fl_dev_mv_fused_supported((int)wq->type, n_embd, 3 * n_embd) && fl_dev_mv_fused_supported((int)wo->type, n_embd, n_embd) &&
           fl_dev_mv_fused_supported((int)w1->type, n_embd, 2 * n_ff) && fl_dev_mv_fused_supported((int)w2->type, n_ff, n_embd));

        if (world > 1) PM(n_head % world == 0 && n_ff % (32 * world) == 0 && (n_embd / world) % 32 == 0 && g->nodes[g->n_nodes - 1]->ne[0] % (2 * world) == 0);
        if (il == 0) {
            ensure_ws(W, n_embd, n_ff, (int)g->nodes[g->n_nodes - 1]->ne[0]);
            P.emb_ids = W.d_tok; P.emb_dst = W.xa;
            xin = W.xa; xout = W.xb;
        }
        PM(W.n_ff == n_ff);
        L.q = W.q;
        L.kcache = dp<const float>(Kv, ctx);
        O.kv_host = Kv->data;
        L.vcache = dp<const float>(Vv, ctx);
        L.att = W.att;
        // wq|wk|wv: rms_norm prologue, rope + cache-store epilogue
        mv_base(L.qkv, (int)wq->type, n_embd);
        L.qkv.nseg = 3;
        const int nl_rows = n_embd / world;                              // this rank's rows of wq / wk / wv (whole heads)
        L.qkv.seg_w[0] = wrows(wq, rank * nl_rows, nl_rows); L.qkv.seg_w[1] = wrows(wk, rank * nl_rows, nl_rows); L.qkv.seg_w[2] = wrows(wv, rank * nl_rows, nl_rows);
        L.qkv.seg_rows[0] = L.qkv.seg_rows[1] = L.qkv.seg_rows[2] = n_embd;
        L.qkv.seg_dst[0] = (float *)L.q;
        L.qkv.pro = FL_PRO_RMSNORM; L.qkv.x = xin; L.qkv.gamma = (const float *)wfull(b->src0);
        L.qkv.epi = FL_EPI_QKV; L.qkv.n_ctx = n_ctx; L.qkv.n_embd = n_embd; L.qkv.head_dim = hd;
        L.qkv.kcache = (float *)L.kcache; L.qkv.vcache = (float *)L.vcache;
        // wo: plain prologue, residual epilogue
        mv_base(L.wo, (int)wo->type, n_embd);
        L.wo.nseg = 1; L.wo.seg_w[0] = world == 1 ? wfull(wo) : nullptr; L.wo.seg_rows[0] = n_embd; L.wo.seg_dst[0] = W.ff;
        L.wo.pro = FL_PRO_PLAIN; L.wo.x = L.att; L.wo.epi = FL_EPI_RESADD; L.wo.res = xin;
        // w1|w3: rms_norm prologue
        mv_base(L.w13, (int)w1->type, n_embd);
        const int fl_rows = n_ff / world;
        L.w13.nseg = 2; L.w13.seg_w[0] = wrows(w1, rank * fl_rows, fl_rows); L.w13.seg_w[1] = wrows(w3, rank * fl_rows, fl_rows);
        L.w13.seg_rows[0] = L.w13.seg_rows[1] = n_ff; L.w13.seg_dst[0] = W.m1; L.w13.seg_dst[1] = W.m3;
        L.w13.pro = FL_PRO_RMSNORM; L.w13.x = W.ff; L.w13.gamma = (const float *)wfull(d->src0); L.w13.epi = FL_EPI_STORE;
        // w2: silu*mul prologue, residual epilogue
        mv_base(L.w2, (int)w2->type, n_ff);
        L.w2.nseg = 1; L.w2.seg_w[0] = world == 1 ? wfull(w2) : nullptr; L.w2.seg_rows[0] = n_embd; L.w2.seg_dst[0] = xout;
        L.w2.pro = FL_PRO_SILUMUL; L.w2.x = L.w13.seg_dst[0]; L.w2.b = L.w13.seg_dst[1]; L.w2.epi = FL_EPI_RESADD; L.w2.res = L.w13.x;
        if (world > 1) {
            // ---- tensor-parallel wiring (SURVEY.md 8e): EVERY matrix is row-split -- wq/wk/wv by heads, w1/w3 by n_ff slices, wo/w2 and
            // the output matrix by output rows -- and every activation vector is all-gathered as a dataflow (LL) vector (make_token_plan).
            // No K-split: a row is always summed over the whole K on one GPU, in the reference's order, so N GPUs produce the bits of one.
            const int nl = n_embd / world, fl = n_ff / world;
            L.kcache += (size_t)rank * nl; L.vcache += (size_t)rank * nl * n_ctx;   // this rank's heads
            for (int i = 0; i < 3; i++) L.qkv.seg_rows[i] = nl;                         // seg_w[] already point at this rank's rows (wrows)
            L.qkv.kcache = (float *)L.kcache; L.qkv.vcache = (float *)L.vcache;
            L.wo.seg_w[0] = wrows(wo, rank * nl, nl); L.wo.seg_rows[0] = nl;
            L.w13.seg_rows[0] = L.w13.seg_rows[1] = fl;
            L.w2.seg_w[0] = wrows(w2, rank * nl, nl); L.w2.seg_rows[0] = nl;
        }
        x = xo;
        std::swap(xin, xout);
    }
    ggml_tensor *e = c.next(GGML_OP_RMS_NORM), *f = c.next(GGML_OP_MUL), *lg = c.next(GGML_OP_MUL_MAT);
    PM(c.ok && c.i == g->n_nodes && e->src0 == x && f->src1 == e && is_vec(f->src0, n_embd) && is_qw(lg->src0) && lg->src1 == f &&
       lg->src0->ne[0] == n_embd && lg->src0->ne[1] % 2 == 0 && fl_dev_mv_fused_supported((int)lg->src0->type, n_embd, (int)lg->src0->ne[1]));
    mv_base(P.head, (int)lg->src0->type, n_embd);
    P.head.nseg = 1; P.head.seg_w[0] = wrows(lg->src0, rank * (int)(lg->src0->ne[1] / world), (int)(lg->src0->ne[1] / world)); P.head.seg_rows[0] = (int)lg->src0->ne[1]; P.head.seg_dst[0] = W.logits;
    PM(W.n_vocab == (int)lg->src0->ne[1] && is_vec(lg, W.n_vocab) && is_vec(f, n_embd));
    P.head.pro = FL_PRO_RMSNORM; P.head.x = xin; P.head.gamma = (const float *)wfull(f->src0); P.head.normed_out = W.emb;
    O.logits_host = lg->data; O.logits_bytes = (size_t)W.n_vocab * 4; O.emb_host = f->data; O.emb_bytes = (size_t)n_embd * 4;
    P.world = world; P.heads_local = n_head / world;
    if (world > 1) {
        PM(W.n_vocab % (2 * world) == 0);
        const int vl = W.n_vocab / world;
        P.head.seg_rows[0] = vl; P.head.seg_dst[0] = W.logits_local;                 // seg_w[0] already points at this rank's rows
        P.vocab_local = vl; P.logits_local = W.logits_local; P.logits_all = W.logits;
    }
    P.head.epi = FL_EPI_STORE;
    P.n_head = n_head; P.n_ctx = n_ctx; P.n_past = n_past;
    return n_past >= 0;
}

bool same_mv(const fl_mv_args &a, const fl_mv_args &b) { return memcmp(&a, &b, sizeof(a)) == 0; }
bool same_plan(const DecodePlan &a, const DecodePlan &b) {
    if (a.n_layer != b.n_layer || a.n_embd != b.n_embd || a.n_head != b.n_head || a.n_ctx != b.n_ctx || a.scale != b.scale ||
        a.emb_type != b.emb_type || a.emb_w != b.emb_w || a.emb_stride != b.emb_stride || a.emb_ids != b.emb_ids || a.emb_dst != b.emb_dst ||
        !same_mv(a.head, b.head) || a.world != b.world)
        return false;
    for (int i = 0; i < a.n_layer; i++) {
        const LayerPlan &x = a.layers[i], &y = b.layers[i];
        if (!same_mv(x.qkv, y.qkv) || !same_mv(x.wo, y.wo) || !same_mv(x.w13, y.w13) || !same_mv(x.w2, y.w2) || x.q != y.q || x.kcache != y.kcache ||
            x.vcache != y.vcache || x.att != y.att)
            return false;
    }
    return true;
}

void profiled_mv(const fl_mv_args &a) {
    if (!g_profile) { FLC(fl_dev_mv_fused(&a)); return; }
    FLC(fl_event_record(g_pev0));
    FLC(fl_dev_mv_fused(&a));
    FLC(fl_event_record(g_pev1));
    FLC(fl_event_sync(g_pev1));
    float ms = 0.f;
    FLC(fl_event_elapsed_ms(g_pev0, g_pev1, &ms));
    int M = 0;
    for (int i = 0; i < a.nseg; i++) M += a.seg_rows[i];
    ggml_b200_kernel_stat *e = nullptr;
    for (auto &k : g_kstats) if (k.type == a.type && k.M == M && k.K == a.K && k.N == 1) e = &k;
    if (!e) {
        g_kstats.push_back(ggml_b200_kernel_stat{a.type, M, a.K, 1, 0, 0.0, (double)M * (a.K / 32) * (double)k_tsize[a.type] + (double)(a.K / 32) * 40.0 + 4.0 * M});
        e = &g_kstats.back();
    }
    e->launches++;
    e->total_ms += ms;
}

// One kernel per matrix group (round 1's path; one GPU only; its dot products add the block terms in another fp32 order than the
// reference, so it only runs on request: FASTLLAMA_B200_MULTI_KERNEL=1).
void issue_decode(const DecodePlan &P, const int *d_npast) {
    FLC(fl_dev_dequantize_rows(P.emb_type, P.emb_w, P.emb_stride, P.emb_K, P.emb_ids, 1, P.emb_dst, (size_t)P.emb_K));
    const int hd = P.n_embd / P.n_head;
    for (const LayerPlan &Lc : P.layers) {
        fl_mv_args qkv = Lc.qkv;
        qkv.n_past = d_npast;
        profiled_mv(qkv);
        FLC(fl_dev_attn_decode(Lc.q, Lc.kcache, Lc.vcache, Lc.att, d_npast, P.n_embd, P.heads_local, hd, P.n_ctx, P.scale));
        profiled_mv(Lc.wo);
        profiled_mv(Lc.w13);
        profiled_mv(Lc.w2);
    }
    profiled_mv(P.head);
}

// The decode step as the program of the persistent token kernel (one cooperative launch per token; fl_token_kernel.cu).
// The activation vectors between the steps -- X: residual stream, A: attention output, B: x + wo.att, H: FFN hidden -- live in one buffer.
//   * one GPU: plain f32 vectors, a grid barrier in front of every step.  (The dataflow form below was measured here too,
//     FASTLLAMA_B200_DATAFLOW=1: 472 vs 550 tokens/s on 7B -- 148 CTAs polling the same words cost more than the barrier they replace.)
//   * `world` GPUs: every matrix is row-split and a step stores its row slice into ALL ranks' copies of the vector as dataflow (LL)
//     words {value, epoch}; the consumer polls for this token's epoch, so no barrier -- local or cross-GPU -- separates the steps
//     (only the one in front of the attention remains: q and the new KV rows of the local CTAs).  The gathered vectors, and with
//     them every later operation, are bit-identical to the one-GPU run.
// Returns nullptr when the shapes are outside what the kernel handles.
void *make_token_plan(const DecodePlan &P, const DecodeWs &W, const int *d_npast) {
    std::vector<fl_token_step> steps;
    const int rank = P.world > 1 ? fl_comm_rank() : 0, world = P.world;
    static const bool dataflow_env = getenv("FASTLLAMA_B200_DATAFLOW") != nullptr;
    const int ll = (world > 1 || dataflow_env) ? 1 : 0;
    const size_t es = ll ? 2 : 1;                                   // floats per element
    const int E = P.n_embd, F = W.n_ff, nl = E / world, fl = F / world, hd = E / P.n_head;
    // element `first` of vector v (0 X, 1 A, 2 B, 3 H) in rank q's buffer, as mapped here
    auto vec = [&](int q, int v, size_t first) -> float * {
        const size_t off = 4096 + (size_t)(v < 3 ? v : 3) * W.ll_cap_embd * 8;
        return (float *)((char *)W.peers[q] + off) + es * first;
    };
    auto peers_of = [&](int v, size_t first, float **dst, int &n) {
        n = 0;
        for (int q = 0; q < world; q++)
            if (q != rank) dst[n++] = vec(q, v, first);
    };
    enum { VX = 0, VA = 1, VB = 2, VH = 3 };
    for (int il = 0; il < P.n_layer; il++) {
        const LayerPlan &Lc = P.layers[il];
        const int seq0 = 4 * il;                                    // A: seq0, B: seq0 + 1, H: seq0 + 2, X (input of layer il + 1): seq0 + 3
        fl_token_step s;
        // wq|wk|wv (this rank's heads): x = embedding row (layer 0) or the residual stream
        memset(&s, 0, sizeof(s));
        s.kind = 0; s.mv = Lc.qkv; s.mv.n_past = d_npast; s.mv.xadd = nullptr; s.mv.sum_out = nullptr;
        if (il == 0) s.mv.x = W.xa;
        else { s.mv.x = vec(rank, VX, 0); s.mv.x_ll = ll; s.mv.x_seq = seq0 - 1; }
        steps.push_back(s);
        // attention over this rank's heads -> elements [rank * nl, +nl) of A (everywhere)
        memset(&s, 0, sizeof(s));
        s.kind = 1; s.q = Lc.q; s.kcache = Lc.kcache; s.vcache = Lc.vcache; s.n_past = d_npast;
        s.k_row_stride = E; s.n_head = P.heads_local; s.head_dim = hd; s.n_ctx = P.n_ctx; s.scale = P.scale;
        s.out = vec(rank, VA, (size_t)rank * nl); s.out_ll = ll; s.out_seq = seq0;
        peers_of(VA, (size_t)rank * nl, s.out_peer, s.n_out_peer);
        steps.push_back(s);
        // wo rows [rank * nl, +nl): B = wo . A + x
        memset(&s, 0, sizeof(s));
        s.kind = 0; s.mv = Lc.wo; s.mv.xadd = nullptr; s.mv.sum_out = nullptr; s.mv.row_stride_bytes = 0;
        s.mv.K = E; s.mv.pro = FL_PRO_PLAIN; s.mv.x = vec(rank, VA, 0); s.mv.x_ll = ll; s.mv.x_seq = seq0;
        s.mv.epi = FL_EPI_RESADD;
        if (il == 0) { s.mv.res = W.xa + (size_t)rank * nl; s.mv.res_ll = 0; }
        else { s.mv.res = vec(rank, VX, (size_t)rank * nl); s.mv.res_ll = ll; }
        s.mv.seg_dst[0] = vec(rank, VB, (size_t)rank * nl); s.mv.out_ll = ll; s.mv.out_seq = seq0 + 1;
        peers_of(VB, (size_t)rank * nl, s.mv.dst_peer, s.mv.n_dst_peer);
        steps.push_back(s);
        // w1|w3 rows [rank * fl, +fl): H = silu(w1 . n) * (w3 . n), n = rms_norm(B) * gamma
        memset(&s, 0, sizeof(s));
        s.kind = 0; s.mv = Lc.w13; s.mv.xadd = nullptr; s.mv.sum_out = nullptr;
        s.mv.x = vec(rank, VB, 0); s.mv.x_ll = ll; s.mv.x_seq = seq0 + 1;
        s.mv.swiglu = 1; s.mv.seg_dst[0] = vec(rank, VH, (size_t)rank * fl); s.mv.seg_dst[1] = nullptr; s.mv.out_ll = ll; s.mv.out_seq = seq0 + 2;
        peers_of(VH, (size_t)rank * fl, s.mv.dst_peer, s.mv.n_dst_peer);
        steps.push_back(s);
        // w2 rows [rank * nl, +nl): X = w2 . H + B
        memset(&s, 0, sizeof(s));
        s.kind = 0; s.mv = Lc.w2; s.mv.xadd = nullptr; s.mv.sum_out = nullptr; s.mv.row_stride_bytes = 0;
        s.mv.K = F; s.mv.pro = FL_PRO_PLAIN; s.mv.b = nullptr; s.mv.x = vec(rank, VH, 0); s.mv.x_ll = ll; s.mv.x_seq = seq0 + 2;
        s.mv.epi = FL_EPI_RESADD; s.mv.res = vec(rank, VB, (size_t)rank * nl); s.mv.res_ll = ll;
        s.mv.seg_dst[0] = vec(rank, VX, (size_t)rank * nl); s.mv.out_ll = ll; s.mv.out_seq = seq0 + 3;
        peers_of(VX, (size_t)rank * nl, s.mv.dst_peer, s.mv.n_dst_peer);
        steps.push_back(s);
    }
    {
        fl_token_step s;
        memset(&s, 0, sizeof(s));
        s.kind = 0; s.mv = P.head; s.mv.xadd = nullptr; s.mv.sum_out = nullptr;
        s.mv.x = vec(rank, VX, 0); s.mv.x_ll = ll; s.mv.x_seq = 4 * P.n_layer - 1;
        steps.push_back(s);
    }
    void *plan = nullptr;
    if (fl_token_plan_create_ll(steps.data(), (int)steps.size(), (unsigned *)W.peers[rank], &plan) != 0) {
        if (g_verbose) fprintf(stderr, "[ggml_b200] token kernel not used: %s\n", fl_last_error());
        return nullptr;
    }
    return plan;
}
void issue_decode_token_kernel(const DecodePlan &P, void *token_plan) {
    FLC(fl_dev_dequantize_rows(P.emb_type, P.emb_w, P.emb_stride, P.emb_K, P.emb_ids, 1, P.emb_dst, (size_t)P.emb_K));
    FLC(fl_token_plan_launch(token_plan));
    if (P.world > 1) FLC(fl_comm_allgather_f32(P.logits_local, P.logits_all, (size_t)P.vocab_local));
}

// returns true when the graph was executed through the fused plan
bool run_decode_plan(const ggml_context *ctx, ggml_cgraph *g, DecodeOutputs &O, void *ev0, void *ev1) {
    DecodeState &D = g_dec;
    if (!D.inited) {
        D.inited = true;
        D.enabled = getenv("FASTLLAMA_B200_NO_FUSED") == nullptr;
        D.use_graph = getenv("FASTLLAMA_B200_NO_GRAPH") == nullptr;
        D.use_token_kernel = getenv("FASTLLAMA_B200_NO_TOKEN_KERNEL") == nullptr;
    }
    if (!D.enabled) return false;
    DecodePlan P;
    const int64_t t_m0 = ggml_time_us();
    if (!match_decode(ctx, g, P, D.ws, O)) return false;
    g_hostprof[1] += (double)(ggml_time_us() - t_m0);
    if (!D.d_npast) {
        D.d_npast = (int *)fl_dev_malloc(64);
        D.h_scalars = (int *)fl_host_alloc_pinned(64);
        if (!D.d_npast || !D.h_scalars) B200_FAIL("decode plan: %s", fl_last_error());
    }
    FLC(fl_dev_rope_table(P.n_embd / P.n_head, P.n_ctx));
    FLC(fl_sync());                                   // the pinned scalars of the previous step have been consumed
    D.h_scalars[0] = P.n_past;
    D.h_scalars[1] = O.token;
    FLC(fl_h2d(D.d_npast, &D.h_scalars[0], sizeof(int)));
    FLC(fl_h2d(D.ws.d_tok, &D.h_scalars[1], sizeof(int)));
    // The persistent token kernel adds every fp32 term in the reference's order (fl_exact.cuh); the one-kernel-per-matrix-group path of
    // round 1 (k_mv_fused / k_attn_decode) does not, so it only runs on request (FASTLLAMA_B200_MULTI_KERNEL=1, measurements) or
    // across GPUs without peer mapping.  A graph the token kernel cannot take is executed node by node (reference order as well).
    static const bool legacy_env = getenv("FASTLLAMA_B200_MULTI_KERNEL") != nullptr;
    const bool legacy = legacy_env || !D.use_token_kernel || (P.world > 1 && !D.ws.peer_mapped);
    const bool eager = g_profile || !D.use_graph;
    if (!same_plan(P, D.plan) || (!legacy && P.world == 1 && !D.token_plan && !D.no_token_plan) || (!eager && !D.graph && !D.no_token_plan)) {
        if (D.graph) { FLC(fl_sync()); FLC(fl_graph_destroy(D.graph)); D.graph = nullptr; }
        if (D.token_plan) { FLC(fl_sync()); FLC(fl_token_plan_destroy(D.token_plan)); D.token_plan = nullptr; }
        D.no_token_plan = false;
        if (!legacy) {
            D.token_plan = make_token_plan(P, D.ws, D.d_npast);
            D.no_token_plan = D.token_plan == nullptr && P.world == 1;      // across GPUs the weights are sharded: the multi-kernel path takes over
        }
        D.plan = P;
        if (P.world > 1) {
            // The ranks reach their first step of a new plan at different times (shard uploads, page faults of an mmap'ed model), but the
            // token kernel's polls for the other ranks' vector elements give up after 2 s: line the ranks up first (one tiny collective).
            FLC(fl_comm_allreduce_f32(D.ws.m3, 1));
            FLC(fl_sync());
        }
        if (!D.no_token_plan) {
            // one eager pass first: sets kernel attributes, and gives this token's result
            FLC(fl_event_record(ev0));
            if (D.token_plan) issue_decode_token_kernel(P, D.token_plan); else issue_decode(P, D.d_npast);
            FLC(fl_event_record(ev1));
            if (!eager) {
                FLC(fl_graph_begin_capture());
                if (D.token_plan) issue_decode_token_kernel(P, D.token_plan); else issue_decode(P, D.d_npast);
                FLC(fl_graph_end_capture(&D.graph));
            }
            g_decode_mode = D.token_plan ? 2 : 1;
            if (g_verbose) fprintf(stderr, "[ggml_b200] decode plan %s: %d layers, n_embd %d, n_ctx %d, %s\n", eager ? "built" : "captured", P.n_layer, P.n_embd, P.n_ctx,
                                   D.token_plan ? "persistent token kernel" : "one kernel per matrix group");
            return true;       // the eager pass already produced this token (capture does not execute)
        }
    }
    if (D.no_token_plan) return false;          // node by node
    if (eager) {
        FLC(fl_event_record(ev0));
        if (D.token_plan) issue_decode_token_kernel(P, D.token_plan); else issue_decode(P, D.d_npast);
        FLC(fl_event_record(ev1));
        g_decode_mode = D.token_plan ? 2 : 1;
        return true;
    }
    FLC(fl_event_record(ev0));
    FLC(fl_graph_launch(D.graph));
    FLC(fl_event_record(ev1));
    g_decode_mode = D.token_plan ? 2 : 1;
    g_stats.graph_replays++;
    return true;
}
}  // namespace

static void decode_state_release() {
    DecodeState &D = g_dec;
    if (!fl_is_initialized()) return;
    if (D.graph) { fl_graph_destroy(D.graph); D.graph = nullptr; }
    if (D.token_plan) { fl_token_plan_destroy(D.token_plan); D.token_plan = nullptr; }
    if (D.ws.xa) {
        fl_dev_free(D.ws.xa);
        if (D.ws.ll_local) fl_dev_free(D.ws.ll_local);
        DecodeWs keep;                                   // the peer-mapped vectors (tensor parallel) stay: they are per process
        if (D.ws.peer_mapped) { memcpy(keep.peers, D.ws.peers, sizeof(keep.peers)); keep.peer_mapped = true; keep.ll_cap_embd = D.ws.ll_cap_embd; keep.ll_cap_ff = D.ws.ll_cap_ff; }
        D.ws = keep;
    }
    D.plan = DecodePlan();
    D.no_token_plan = false;
    D.tp_kv_sharded = false;
    g_tp_kv_sharded = false;
    if (g_exec.q8_work) { fl_dev_free(g_exec.q8_work); g_exec.q8_work = nullptr; g_exec.q8_cap = 0; }
}

// Tensor-parallel decode steps write only this rank's heads of the new positions into the KV cache (K [pos][n_embd]: nl
// columns per row; V [n_embd][n_ctx]: nl rows).  Before anything reads the cache as a whole -- a replicated multi-token
// eval, save_state -- the ranks exchange those slices: pack (strided copies) -> one all-gather -> unpack.  Collective.
static void tp_gather_kv() {
    DecodeState &D = g_dec;
    const DecodePlan &P = D.plan;
    const int world = fl_comm_world(), rank = fl_comm_rank();
    if (!D.tp_kv_sharded || world <= 1 || P.layers.empty()) { D.tp_kv_sharded = false; g_tp_kv_sharded = false; return; }
    const int npos = D.tp_end_pos - D.tp_first_pos, first = D.tp_first_pos;
    const int n_embd = P.n_embd, n_ctx = P.n_ctx, nl = n_embd / world, L = (int)P.layers.size();
    const size_t per_layer = (size_t)2 * npos * nl, count = per_layer * L;
    float *send = (float *)fl_dev_malloc(count * sizeof(float) * (size_t)(world + 1));
    if (!send) B200_FAIL("KV gather: %s", fl_last_error());
    float *recv = send + count;
    for (int l = 0; l < L; l++) {
        const float *kmine = P.layers[l].kcache + (size_t)first * n_embd;                  // already offset to this rank's columns
        const float *vmine = P.layers[l].vcache + first;                                   // already offset to this rank's rows
        FLC(fl_d2d_2d(send + l * per_layer, (size_t)nl * 4, kmine, (size_t)n_embd * 4, (size_t)nl * 4, (size_t)npos));
        FLC(fl_d2d_2d(send + l * per_layer + (size_t)npos * nl, (size_t)npos * 4, vmine, (size_t)n_ctx * 4, (size_t)npos * 4, (size_t)nl));
    }
    FLC(fl_comm_allgather_f32(send, recv, count));
    for (int r = 0; r < world; r++) {
        if (r == rank) continue;
        for (int l = 0; l < L; l++) {
            float *kbase = (float *)P.layers[l].kcache - (size_t)rank * nl;                // the layer's K [pos][n_embd]
            float *vbase = (float *)P.layers[l].vcache - (size_t)rank * nl * n_ctx;        // the layer's V [n_embd][n_ctx]
            const float *src = recv + (size_t)r * count + l * per_layer;
            FLC(fl_d2d_2d(kbase + (size_t)first * n_embd + (size_t)r * nl, (size_t)n_embd * 4, src, (size_t)nl * 4, (size_t)nl * 4, (size_t)npos));
            FLC(fl_d2d_2d(vbase + (size_t)r * nl * n_ctx + first, (size_t)n_ctx * 4, src + (size_t)npos * nl, (size_t)npos * 4, (size_t)npos * 4, (size_t)nl));
        }
    }
    FLC(fl_sync());
    FLC(fl_dev_free(send));
    if (g_verbose) fprintf(stderr, "[ggml_b200] gathered the KV cache of positions [%d, %d) from %d ranks\n", first, D.tp_end_pos, world);
    D.tp_kv_sharded = false;
    g_tp_kv_sharded = false;
}

extern "C" void ggml_graph_compute(struct ggml_context *ctx, struct ggml_cgraph *g) {
    ensure_backend();
    static void *ev0 = nullptr, *ev1 = nullptr;
    if (!ev0) { ev0 = fl_event_create(); ev1 = fl_event_create(); }
    const int64_t t_start = ggml_time_us();
    static const bool sync_all = getenv("FASTLLAMA_B200_SYNC_ALL") != nullptr;

    g->work = nullptr;
    g->work_size = 0;

    DecodeOutputs dout;
    const int64_t t_in = ggml_time_us();
    if (run_decode_plan(ctx, g, dout, ev0, ev1)) {
        const int64_t t_issued = ggml_time_us();
        mark_device_write(dout.kv_host, ctx);          // the step appended one position to the KV cache on the device
        if (fl_comm_world() > 1) {
            const int pos = g_dec.h_scalars[0];                   // n_past of this step = the position it wrote
            if (!g_dec.tp_kv_sharded) { g_dec.tp_first_pos = pos; g_dec.tp_end_pos = pos + 1; }
            else { g_dec.tp_first_pos = std::min(g_dec.tp_first_pos, pos); g_dec.tp_end_pos = std::max(g_dec.tp_end_pos, pos + 1); }
            g_dec.tp_kv_sharded = true; g_tp_kv_sharded = true;
        }
        // fused decode step: the two results the caller reads (reference lib/llama.cpp:476-489) come
        // straight from the private workspace
        // through pinned staging: a device-to-host copy into the caller's pageable arena would be staged by the driver, synchronously
        if (g_dec.h_out_cap < dout.logits_bytes + dout.emb_bytes) {
            if (g_dec.h_out) FLC(fl_host_free_pinned(g_dec.h_out));
            g_dec.h_out_cap = dout.logits_bytes + dout.emb_bytes;
            g_dec.h_out = (char *)fl_host_alloc_pinned(g_dec.h_out_cap);
            if (!g_dec.h_out) B200_FAIL("decode result staging: %s", fl_last_error());
        }
        FLC(fl_d2h(g_dec.h_out, g_dec.ws.logits, dout.logits_bytes));
        FLC(fl_d2h(g_dec.h_out + dout.logits_bytes, g_dec.ws.emb, dout.emb_bytes));
        FLC(fl_sync());
        memcpy(dout.logits_host, g_dec.h_out, dout.logits_bytes);
        memcpy(dout.emb_host, g_dec.h_out + dout.logits_bytes, dout.emb_bytes);
        if (g_dec.token_plan && fl_token_plan_error(g_dec.token_plan))
            B200_FAIL("%s", fl_last_error());
        const int64_t t_out = ggml_time_us();
        g_hostprof[0] += 1;
        g_hostprof[2] += (double)(t_issued - t_in);          // includes [1]
        g_hostprof[3] += (double)(t_out - t_issued);
        if (g_last_exit_us) g_hostprof[4] += (double)(t_in - g_last_exit_us);
        g_last_exit_us = t_out;
    } else {
        g_last_exit_us = 0;
        g_decode_mode = 0;
        // Leafs.  Weights / KV cache live in persistent arenas (uploaded once by dev_ptr).  Constants the
        // host wrote into the compute arena while building the graph are uploaded per graph, but only
        // those a device op reads as DATA (token ids); rope / mask / scale parameters are read on the
        // host at dispatch, so ~130 tiny copies per 7B token are avoided.
        {
            const ggml_tensor *done[16];
            int n_done = 0;
            auto upload_leaf = [&](const ggml_tensor *t) {
                if (!t || t->op != GGML_OP_NONE || !t->data || !in_ctx(ctx, t->data)) return;
                for (int i = 0; i < n_done; i++) if (done[i] == t) return;
                const size_t nb = nbytes_of(t);
                FLC(fl_h2d(dev_ptr(t->data, nb, ctx), t->data, nb));
                if (n_done < 16) done[n_done++] = t;
            };
            for (int i = 0; i < g->n_nodes; i++) {
                const ggml_tensor *n = g->nodes[i];
                const bool param_only = n->op == GGML_OP_SCALE || n->op == GGML_OP_DIAG_MASK_INF || n->op == GGML_OP_ROPE;
                upload_leaf(n->src0);
                if (!param_only) upload_leaf(n->src1);
            }
        }

        if (g_dec.tp_kv_sharded)
            for (int i = 0; i < g->n_nodes; i++)
                if (g->nodes[i]->op == GGML_OP_SOFT_MAX) { tp_gather_kv(); break; }    // a replicated attention eval needs every head's K/V
        FLC(fl_event_record(ev0));
        for (int i = 0; i < g->n_nodes; i++) exec_node(g->nodes[i], ctx);
        FLC(fl_event_record(ev1));

        // results the caller may read on the host (reference lib/llama.cpp:476-489): graph sinks that
        // live in the compute arena (the logits) and the input of the last mul_mat (the embeddings).
        std::vector<char> consumed((size_t)g->n_nodes, 0);
        {
            const GraphEpoch *ge = lookup_epoch(g);
            const bool by_stamp = ge && ge->clean && ge->epoch == g_epoch;
            std::unordered_map<const ggml_tensor *, int> index;
            if (!by_stamp)
                for (int i = 0; i < g->n_nodes; i++) index[g->nodes[i]] = i;
            auto mark = [&](const ggml_tensor *s) {
                if (!s) return;
                if (by_stamp) {
                    const Stamp *st = (const Stamp *)s->padding;
                    if (st->epoch == ge->epoch && st->index >= 0 && st->index < g->n_nodes && g->nodes[st->index] == s) consumed[st->index] = 1;
                } else {
                    auto it = index.find(s);
                    if (it != index.end()) consumed[it->second] = 1;
                }
            };
            for (int i = 0; i < g->n_nodes; i++) {
                mark(g->nodes[i]->src0); mark(g->nodes[i]->src1);
                for (int k = 0; k < GGML_MAX_OPT; k++) mark(g->nodes[i]->opt[k]);
            }
        }
        const ggml_tensor *last_mm = nullptr;
        for (int i = g->n_nodes - 1; i >= 0 && !last_mm; i--)
            if (g->nodes[i]->op == GGML_OP_MUL_MAT) last_mm = g->nodes[i];
        for (int i = 0; i < g->n_nodes; i++) {
            ggml_tensor *t = g->nodes[i];
            const bool want = sync_all || !consumed[i] || (last_mm && t == last_mm->src1);
            if (!want || !in_ctx(ctx, t->data) || !is_contiguous(t)) continue;
            const size_t nb = nbytes_of(t);
            FLC(fl_d2h(t->data, dev_ptr(t->data, nb, ctx), nb));
        }
        FLC(fl_sync());
    }

    float ms = 0.f;
    FLC(fl_event_elapsed_ms(ev0, ev1, &ms));
    g_stats.n_evals++;
    g_stats.last_us = ms * 1000.0;
    g_stats.total_us += ms * 1000.0;
    g->perf_runs++;
    g->perf_time_us += ggml_time_us() - t_start;
}

// ================================================================================================
// quantisation entry points (model-file creation, test hook) -- all on the GPU
// ================================================================================================
static void hist_add(const uint8_t *blocks, size_t nblocks, size_t bb, size_t qoff, int64_t *hist) {
    if (!hist) return;
    for (size_t i = 0; i < nblocks; i++) {
        const uint8_t *qs = blocks + i * bb + qoff;
        for (int j = 0; j < 16; j++) { hist[qs[j] & 0xF]++; hist[qs[j] >> 4]++; }
    }
}
extern "C" size_t ggml_quantize_q4_0(const float *src, void *dst, int n, int k, int64_t *hist) {
    ensure_backend();
    B200_ASSERT(k % 32 == 0 && n % k == 0);
    FLC(fl_quantize_rows_q4(FL_Q4_0, src, dst, k, n / k));
    hist_add((const uint8_t *)dst, (size_t)n / 32, 20, 4, hist);
    return (size_t)n / 32 * 20;
}
extern "C" size_t ggml_quantize_q4_1(const float *src, void *dst, int n, int k, int64_t *hist) {
    ensure_backend();
    B200_ASSERT(k % 32 == 0 && n % k == 0);
    FLC(fl_quantize_rows_q4(FL_Q4_1, src, dst, k, n / k));
    hist_add((const uint8_t *)dst, (size_t)n / 32, 24, 8, hist);
    return (size_t)n / 32 * 24;
}
extern "C" size_t ggml_quantize_chunk(enum ggml_type type, const float *src, void *dst, int start, int n, int64_t *hist) {
    B200_ASSERT(start % 32 == 0);
    switch (type) {
        case GGML_TYPE_Q4_0: return ggml_quantize_q4_0(src + start, (char *)dst + (size_t)start / 32 * 20, n, n, hist);
        case GGML_TYPE_Q4_1: return ggml_quantize_q4_1(src + start, (char *)dst + (size_t)start / 32 * 24, n, n, hist);
        default: B200_FAIL("ggml_quantize_chunk: type %s is not supported by the B200 backend (q4_0, q4_1)", k_tname[type]);
    }
}

namespace {
template <int T> void hook_dequantize(const void *x, float *y, int k) { ensure_backend(); FLC(fl_dequantize_rows_q4(T, x, y, k, 1)); }
template <int T> void hook_quantize_ref(const float *x, void *y, int k) { ensure_backend(); FLC(fl_quantize_rows_q4(T, x, y, k, 1)); }
template <int T> void hook_quantize_simd(const float *x, void *y, int k) { ensure_backend(); FLC(fl_quantize_rows_q4_simd(T, x, y, k, 1)); }
void hook_quantize_q8(const float *x, void *y, int k) { ensure_backend(); FLC(fl_quantize_row_q8_0(x, y, k)); }
template <int T> void hook_vec_dot(const int n, float *s, const void *x, const void *y) { ensure_backend(); FLC(fl_vec_dot_q4_q8(T, n, s, x, y)); }
}  // namespace

extern "C" quantize_fns_t ggml_internal_get_quantize_fn(size_t i) {
    quantize_fns_t f = {nullptr, nullptr, nullptr, nullptr, nullptr};
    if (i == GGML_TYPE_Q4_0) f = {hook_dequantize<FL_Q4_0>, hook_quantize_simd<FL_Q4_0>, hook_quantize_ref<FL_Q4_0>, hook_quantize_q8, hook_vec_dot<FL_Q4_0>};
    if (i == GGML_TYPE_Q4_1) f = {hook_dequantize<FL_Q4_1>, hook_quantize_simd<FL_Q4_1>, hook_quantize_ref<FL_Q4_1>, hook_quantize_q8, hook_vec_dot<FL_Q4_1>};
    if (i == GGML_TYPE_Q8_0) f.quantize_row_q = f.quantize_row_q_reference = f.quantize_row_q_dot = hook_quantize_q8;
    return f;
}
