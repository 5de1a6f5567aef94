// Plan-level C entry (SURVEY.md 8(b), last row): the LAUNCH LIST of a program -- one UNet forward, the context program, one whole
// sampler step (next timestep -> UNet -> CFG + DDIM update), a VAE decode ... -- lives behind the C ABI as an `sdk_plan`:
//
//   * the host that plans a program (the Python package) records every launch with sdk_plan_add_launch(): the NAME of a
//     launch-type entry point of sdb200.h plus its arguments widened to 64 bits; tensor-core GEMM / attention / projection+LayerNorm
//     handles are ADOPTED by the plan together with the descriptor they were created from (tuned tiling included), so the plan
//     owns them and can re-create them;
//   * sdk_plan_launch() replays a program in ONE call (optionally as a CUDA graph the plan captured itself);
//   * sdk_plan_save() writes a self-contained ENGINE FILE: every device pointer of every launch / descriptor is rewritten as
//     (memory region, offset), the contents of the constant regions (packed weights, timestep / coefficient tables) follow;
//   * sdk_plan_load() lets ANY host -- no Python, no PyTorch -- allocate the regions, upload the constants, re-create the
//     handles (TMA descriptors are re-encoded for the new addresses) and run the programs: tools/c_host/denoise.c is a C program
//     that runs UNet forwards and the full sampling loop from an engine file through nothing but this header.
//
// The reference has no such layer (its programs are eager PyTorch: models/unet/unet.py:431-443 called from
// models/diffusion.py:223-236); this is the boundary a non-Python serving host binds.
#define SDK_PDL_CAT 8
#include "common.cuh"
#include "../../include/sdb200.h"
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

namespace {

// ---- argument marshalling: uint64 slots -> the C types of a launch-type entry point (the trailing `void* stream` is appended) ----
template <typename T> struct ArgConv;
template <typename T> struct ArgConv<T*> { static constexpr bool is_ptr = true; static T* get(uint64_t v) { return reinterpret_cast<T*>((uintptr_t)v); } };
template <> struct ArgConv<int> { static constexpr bool is_ptr = false; static int get(uint64_t v) { return (int)(int64_t)v; } };
template <> struct ArgConv<int64_t> { static constexpr bool is_ptr = false; static int64_t get(uint64_t v) { return (int64_t)v; } };
template <> struct ArgConv<float> {
    static constexpr bool is_ptr = false;
    static float get(uint64_t v) { const uint32_t b = (uint32_t)v; float f; memcpy(&f, &b, 4); return f; }
};

enum FnKind { FN_PLAIN = 0, FN_HANDLE = 1, FN_STRUCT = 2 };
enum HandleKind { H_TC_GEMM = 1, H_ATTENTION_TC = 2, H_LINEAR_LN = 3 };

struct FnEntry {
    const char* name;
    void* fn;
    int nargs;
    uint32_t ptr_mask;                    // which arguments are DEVICE pointers (relocated by save / load)
    int (*invoke)(void* fn, const uint64_t* a, void* stream);
    int kind, handle_kind;
};

template <typename... Args> struct Sig {
    static constexpr int N = (int)sizeof...(Args) - 1;
    using Tup = std::tuple<Args...>;
    template <size_t... I> static int inv(void* f, const uint64_t* a, void* s, std::index_sequence<I...>) {
        return reinterpret_cast<int (*)(Args...)>(f)(ArgConv<std::tuple_element_t<I, Tup>>::get(a[I])..., s);
    }
    static int invoke(void* f, const uint64_t* a, void* s) { return inv(f, a, s, std::make_index_sequence<N>{}); }
    template <size_t... I> static uint32_t mask(std::index_sequence<I...>) {
        uint32_t m = 0;
        const bool flags[] = {ArgConv<std::tuple_element_t<I, Tup>>::is_ptr..., false};
        for (int i = 0; i < N; ++i) if (flags[i]) m |= 1u << i;
        return m;
    }
};
template <typename... Args> FnEntry entry(const char* name, int (*fn)(Args...), int kind = FN_PLAIN, int hk = 0) {
    static_assert(sizeof...(Args) >= 1 && sizeof...(Args) <= 25, "launch-type entry points take 0..24 arguments and a stream");
    FnEntry e;
    e.name = name; e.fn = reinterpret_cast<void*>(fn); e.nargs = Sig<Args...>::N;
    e.ptr_mask = kind == FN_PLAIN ? Sig<Args...>::mask(std::make_index_sequence<Sig<Args...>::N>{}) : 0u;
    e.invoke = &Sig<Args...>::invoke; e.kind = kind; e.handle_kind = hk;
    return e;
}

#define E(fn) entry(#fn, &fn)
const std::vector<FnEntry>& registry() {
    static const std::vector<FnEntry> r = {
        E(sdk_zero), E(sdk_ddim_step), E(sdk_ddpm_step), E(sdk_ddim_inpaint_step), E(sdk_ddpm_inpaint_step), E(sdk_dpmpp_step),
        E(sdk_dpmpp_inpaint_step), E(sdk_forward_process), E(sdk_x0_from_eps),
        E(sdk_next_timestep), E(sdk_gather_row),
        E(sdk_groupnorm_stats), E(sdk_groupnorm_apply), E(sdk_groupnorm_apply_cs), E(sdk_channel_stats), E(sdk_groupnorm_fused),
        E(sdk_groupnorm_cluster), E(sdk_layernorm), E(sdk_softmax_rows), E(sdk_embed_tokens), E(sdk_activation), E(sdk_cast_upsample),
        E(sdk_nchw_to_nhwc), E(sdk_time_sinusoid), E(sdk_gemv), E(sdk_conv_in), E(sdk_im2col_s2),
        E(sdk_attention_f32), E(sdk_attention_f32_ex), E(sdk_attention_bf16), E(sdk_lora_merge),
        entry("sdk_conv_gemm_f32", &sdk_conv_gemm_f32, FN_STRUCT),
        entry("sdk_tc_gemm_launch", &sdk_tc_gemm_launch, FN_HANDLE, H_TC_GEMM),
        entry("sdk_attention_tc_launch", &sdk_attention_tc_launch, FN_HANDLE, H_ATTENTION_TC),
        entry("sdk_linear_ln_launch", &sdk_linear_ln_launch, FN_HANDLE, H_LINEAR_LN),
    };
    return r;
}
#undef E

int find_fn(const char* name) {
    const auto& r = registry();
    for (size_t i = 0; i < r.size(); ++i) if (strcmp(r[i].name, name) == 0) return (int)i;
    return -1;
}

// ---- device-pointer fields of the descriptors (relocation) ----
const size_t TC_PTRS[] = {offsetof(SdkTcGemmDesc, a), offsetof(SdkTcGemmDesc, a) + sizeof(void*), offsetof(SdkTcGemmDesc, w),
                          offsetof(SdkTcGemmDesc, w) + sizeof(void*), offsetof(SdkTcGemmDesc, bias), offsetof(SdkTcGemmDesc, tbias),
                          offsetof(SdkTcGemmDesc, residual), offsetof(SdkTcGemmDesc, out), offsetof(SdkTcGemmDesc, out2),
                          offsetof(SdkTcGemmDesc, row_stats), offsetof(SdkTcGemmDesc, ln_stats), offsetof(SdkTcGemmDesc, ln_colsum)};
const size_t ATT_PTRS[] = {offsetof(SdkAttentionTcDesc, q), offsetof(SdkAttentionTcDesc, k), offsetof(SdkAttentionTcDesc, v),
                           offsetof(SdkAttentionTcDesc, out)};
const size_t LLN_PTRS[] = {offsetof(SdkLinearLnDesc, a), offsetof(SdkLinearLnDesc, w), offsetof(SdkLinearLnDesc, bias),
                           offsetof(SdkLinearLnDesc, residual), offsetof(SdkLinearLnDesc, out), offsetof(SdkLinearLnDesc, ln_out),
                           offsetof(SdkLinearLnDesc, gamma), offsetof(SdkLinearLnDesc, beta)};
const size_t CONV_PTRS[] = {offsetof(SdkConvParams, src0), offsetof(SdkConvParams, src1), offsetof(SdkConvParams, weight),
                            offsetof(SdkConvParams, bias), offsetof(SdkConvParams, tbias), offsetof(SdkConvParams, residual),
                            offsetof(SdkConvParams, out)};

struct PtrTable { const size_t* off; int n; size_t size; };
PtrTable desc_ptrs(int hk) {
    switch (hk) {
        case H_TC_GEMM: return {TC_PTRS, (int)(sizeof(TC_PTRS) / sizeof(size_t)), sizeof(SdkTcGemmDesc)};
        case H_ATTENTION_TC: return {ATT_PTRS, (int)(sizeof(ATT_PTRS) / sizeof(size_t)), sizeof(SdkAttentionTcDesc)};
        case H_LINEAR_LN: return {LLN_PTRS, (int)(sizeof(LLN_PTRS) / sizeof(size_t)), sizeof(SdkLinearLnDesc)};
    }
    return {nullptr, 0, 0};
}

constexpr int MAX_ARGS = 24, MAX_PROGRAMS = 16;
constexpr uint64_t RELOC_TAG = 0x8000000000000000ull;      // encoded pointer: tag | region << 40 | offset

struct Op { int fn; int nargs; uint64_t args[MAX_ARGS]; int handle; int blob; };
struct HandleRec {
    int kind; std::vector<uint8_t> desc; void* h;
    uint64_t aux[2];              // tc_gemm: {channel-statistics table, split-K workspace} (device pointers); attention: {causal, 0}
};
struct Region { uint64_t base, bytes; int kind; std::string name; bool used; };
struct Plan {
    std::vector<Op> prog[MAX_PROGRAMS];
    std::vector<HandleRec> handles;
    std::vector<Region> regions;
    std::vector<std::vector<uint8_t>> blobs;       // SdkConvParams copies
    void* slab = nullptr;                          // device memory owned by a LOADED plan
    cudaGraphExec_t graph[MAX_PROGRAMS] = {};
    cudaGraph_t graph_src[MAX_PROGRAMS] = {};
};

int destroy_handle(HandleRec& r) {
    if (!r.h) return SDK_OK;
    int rc = SDK_OK;
    if (r.kind == H_TC_GEMM) rc = sdk_tc_gemm_destroy(r.h);
    else if (r.kind == H_ATTENTION_TC) rc = sdk_attention_tc_destroy(r.h);
    else if (r.kind == H_LINEAR_LN) rc = sdk_linear_ln_destroy(r.h);
    r.h = nullptr;
    return rc;
}

int create_handle(HandleRec& r) {
    int rc = SDK_ERR_ARG;
    if (r.kind == H_TC_GEMM) {
        rc = sdk_tc_gemm_create(reinterpret_cast<const SdkTcGemmDesc*>(r.desc.data()), &r.h);
        if (rc == SDK_OK && r.aux[1]) rc = sdk_tc_gemm_set_workspace(r.h, reinterpret_cast<void*>((uintptr_t)r.aux[1]));
        if (rc == SDK_OK && r.aux[0]) rc = sdk_tc_gemm_set_stats(r.h, reinterpret_cast<double*>((uintptr_t)r.aux[0]));
    } else if (r.kind == H_ATTENTION_TC) {
        const SdkAttentionTcDesc* d = reinterpret_cast<const SdkAttentionTcDesc*>(r.desc.data());
        rc = sdk_attention_tc_create(d->q, d->q_row, d->q_batch, d->k, d->k_row, d->k_batch, d->v, d->v_row, d->v_batch, d->out, d->o_row,
                                     d->o_batch, d->B, d->heads, d->Sq, d->Sk, d->D, d->scale, &r.h);
        if (rc == SDK_OK && r.aux[0]) rc = sdk_attention_tc_set_causal(r.h, 1);
    } else if (r.kind == H_LINEAR_LN) {
        rc = sdk_linear_ln_create(reinterpret_cast<const SdkLinearLnDesc*>(r.desc.data()), &r.h);
    }
    return rc;
}

// pointer -> (region, offset)
bool encode_ptr(Plan* p, uint64_t v, uint64_t* out) {
    if (v == 0) { *out = 0; return true; }
    for (size_t i = 0; i < p->regions.size(); ++i) {
        Region& r = p->regions[i];
        if (v >= r.base && v < r.base + r.bytes) {
            r.used = true;
            *out = RELOC_TAG | ((uint64_t)i << 40) | (v - r.base);
            return true;
        }
    }
    return false;
}
uint64_t decode_ptr(const std::vector<uint64_t>& bases, uint64_t v) {
    if (!(v & RELOC_TAG)) return v;
    const uint64_t idx = (v & ~RELOC_TAG) >> 40, off = v & ((1ull << 40) - 1);
    return idx < bases.size() ? bases[idx] + off : 0;
}

struct Writer {
    FILE* f; bool ok = true;
    void raw(const void* d, size_t n) { if (ok && n && fwrite(d, 1, n, f) != n) ok = false; }
    void u32(uint32_t v) { raw(&v, 4); }
    void u64(uint64_t v) { raw(&v, 8); }
    void str(const std::string& s) { u32((uint32_t)s.size()); raw(s.data(), s.size()); }
};
struct Reader {
    FILE* f; bool ok = true;
    void raw(void* d, size_t n) { if (ok && n && fread(d, 1, n, f) != n) ok = false; }
    uint32_t u32() { uint32_t v = 0; raw(&v, 4); return v; }
    uint64_t u64() { uint64_t v = 0; raw(&v, 8); return v; }
    std::string str() { const uint32_t n = u32(); std::string s; if (ok && n < (1u << 20)) { s.resize(n); raw(&s[0], n); } else ok = false; return s; }
};

const char MAGIC[8] = {'S', 'D', 'B', '2', '0', '0', 'P', 'L'};
constexpr uint32_t FILE_VERSION = 1;

}  // namespace

extern "C" int sdk_plan_create(void** plan) {
    SDK_CHECK_ARG(plan, "sdk_plan_create: null pointer");
    Plan* p = new (std::nothrow) Plan();
    if (!p) return sdk_fail(SDK_ERR_CUDA, "out of host memory");
    *plan = p;
    return SDK_OK;
}

extern "C" int sdk_plan_destroy(void* plan) {
    if (!plan) return SDK_OK;
    Plan* p = static_cast<Plan*>(plan);
    for (int i = 0; i < MAX_PROGRAMS; ++i) {
        if (p->graph[i]) cudaGraphExecDestroy(p->graph[i]);
        if (p->graph_src[i]) cudaGraphDestroy(p->graph_src[i]);
    }
    for (auto& h : p->handles) destroy_handle(h);
    if (p->slab) cudaFree(p->slab);
    delete p;
    return SDK_OK;
}

extern "C" int sdk_plan_add_region(void* plan, const void* base, int64_t bytes, int kind, const char* name) {
    SDK_CHECK_ARG(plan && base && bytes > 0 && kind >= 0 && kind <= 2, "sdk_plan_add_region: bad arguments");
    Plan* p = static_cast<Plan*>(plan);
    const uint64_t b = (uint64_t)(uintptr_t)base;
    for (auto& r : p->regions) {
        if (r.base == b && r.bytes == (uint64_t)bytes) {                 // registering a buffer twice is harmless
            if (name && *name && r.name.empty()) r.name = name;
            return SDK_OK;
        }
        if (b < r.base + r.bytes && r.base < b + (uint64_t)bytes)
            return sdk_fail(SDK_ERR_ARG, "sdk_plan_add_region: [%p, +%lld) overlaps region '%s'", base, (long long)bytes, r.name.c_str());
    }
    p->regions.push_back(Region{b, (uint64_t)bytes, kind, name ? name : "", false});
    return SDK_OK;
}

extern "C" int sdk_plan_adopt(void* plan, int handle_kind, void* handle, const void* desc, int desc_bytes, const uint64_t* aux, int n_aux) {
    SDK_CHECK_ARG(plan && handle && desc && n_aux >= 0 && n_aux <= 2, "sdk_plan_adopt: bad arguments");
    const PtrTable t = desc_ptrs(handle_kind);
    SDK_CHECK_ARG(t.size != 0 && (size_t)desc_bytes == t.size, "sdk_plan_adopt: handle kind %d with a %d-byte descriptor", handle_kind, desc_bytes);
    Plan* p = static_cast<Plan*>(plan);
    for (auto& h : p->handles) SDK_CHECK_ARG(h.h != handle, "sdk_plan_adopt: handle adopted twice");
    HandleRec r;
    r.kind = handle_kind; r.h = handle;
    r.desc.assign(static_cast<const uint8_t*>(desc), static_cast<const uint8_t*>(desc) + desc_bytes);
    r.aux[0] = n_aux > 0 ? aux[0] : 0; r.aux[1] = n_aux > 1 ? aux[1] : 0;
    p->handles.push_back(r);
    return SDK_OK;
}

extern "C" int sdk_plan_add_launch(void* plan, int program, const char* fn_name, const uint64_t* args, int nargs) {
    SDK_CHECK_ARG(plan && fn_name && program >= 0 && program < MAX_PROGRAMS && nargs >= 0 && nargs <= MAX_ARGS && (args || nargs == 0),
                  "sdk_plan_add_launch: bad arguments");
    Plan* p = static_cast<Plan*>(plan);
    const int fi = find_fn(fn_name);
    if (fi < 0) return sdk_fail(SDK_ERR_UNSUPPORTED, "sdk_plan_add_launch: '%s' is not a launch-type entry point of sdb200.h", fn_name);
    const FnEntry& e = registry()[fi];
    SDK_CHECK_ARG(nargs == e.nargs, "sdk_plan_add_launch: %s takes %d arguments before the stream, got %d", fn_name, e.nargs, nargs);
    Op op;
    memset(&op, 0, sizeof(op));
    op.fn = fi; op.nargs = nargs; op.handle = -1; op.blob = -1;
    for (int i = 0; i < nargs; ++i) op.args[i] = args[i];
    if (e.kind == FN_HANDLE) {
        for (size_t i = 0; i < p->handles.size(); ++i)
            if ((uint64_t)(uintptr_t)p->handles[i].h == args[0] && p->handles[i].kind == e.handle_kind) op.handle = (int)i;
        SDK_CHECK_ARG(op.handle >= 0, "sdk_plan_add_launch: %s on a handle the plan has not adopted (sdk_plan_adopt)", fn_name);
    } else if (e.kind == FN_STRUCT) {
        SDK_CHECK_ARG(args[0], "sdk_plan_add_launch: %s needs its parameter struct", fn_name);
        const uint8_t* src = reinterpret_cast<const uint8_t*>((uintptr_t)args[0]);
        p->blobs.emplace_back(src, src + sizeof(SdkConvParams));
        op.blob = (int)p->blobs.size() - 1;
    }
    p->prog[program].push_back(op);
    return SDK_OK;
}

extern "C" int sdk_plan_num_launches(void* plan, int program) {
    if (!plan || program < 0 || program >= MAX_PROGRAMS) return -1;
    return (int)static_cast<Plan*>(plan)->prog[program].size();
}

namespace {
int enqueue(Plan* p, int program, void* stream) {
    const auto& reg = registry();
    for (const Op& op : p->prog[program]) {
        const FnEntry& e = reg[op.fn];
        uint64_t a[MAX_ARGS];
        for (int i = 0; i < op.nargs; ++i) a[i] = op.args[i];
        if (e.kind == FN_HANDLE) a[0] = (uint64_t)(uintptr_t)p->handles[op.handle].h;
        else if (e.kind == FN_STRUCT) a[0] = (uint64_t)(uintptr_t)p->blobs[op.blob].data();
        const int rc = e.invoke(e.fn, a, stream);
        if (rc != SDK_OK) return rc;
    }
    return SDK_OK;
}
}  // namespace

extern "C" int sdk_plan_launch(void* plan, int program, void* stream) {
    SDK_CHECK_ARG(plan && program >= 0 && program < MAX_PROGRAMS, "sdk_plan_launch: bad arguments");
    Plan* p = static_cast<Plan*>(plan);
    if (p->graph[program]) { SDK_CUDA(cudaGraphLaunch(p->graph[program], static_cast<cudaStream_t>(stream))); return SDK_OK; }
    return enqueue(p, program, stream);
}

// Capture `program` into a CUDA graph owned by the plan (call after ONE eager sdk_plan_launch of the program on this device: the first
// launch of a kernel sets its function attributes, which is not capturable); later sdk_plan_launch calls replay the graph.
extern "C" int sdk_plan_capture(void* plan, int program, void* stream) {
    SDK_CHECK_ARG(plan && program >= 0 && program < MAX_PROGRAMS && stream, "sdk_plan_capture: needs a plan, a program and a non-default stream");
    Plan* p = static_cast<Plan*>(plan);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (p->graph[program]) { cudaGraphExecDestroy(p->graph[program]); p->graph[program] = nullptr; }
    if (p->graph_src[program]) { cudaGraphDestroy(p->graph_src[program]); p->graph_src[program] = nullptr; }
    SDK_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    const int rc = enqueue(p, program, stream);
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(s, &g);
    if (rc != SDK_OK) { if (g) cudaGraphDestroy(g); return rc; }
    if (e != cudaSuccess) return sdk_fail(SDK_ERR_CUDA, "sdk_plan_capture: cudaStreamEndCapture: %s", cudaGetErrorString(e));
    cudaGraphExec_t ge = nullptr;
    const cudaError_t e2 = cudaGraphInstantiate(&ge, g, 0);
    if (e2 != cudaSuccess) { cudaGraphDestroy(g); return sdk_fail(SDK_ERR_CUDA, "sdk_plan_capture: cudaGraphInstantiate: %s", cudaGetErrorString(e2)); }
    p->graph[program] = ge; p->graph_src[program] = g;
    return SDK_OK;
}

extern "C" int sdk_plan_region(void* plan, const char* name, void** ptr, int64_t* bytes) {
    SDK_CHECK_ARG(plan && name && ptr, "sdk_plan_region: bad arguments");
    Plan* p = static_cast<Plan*>(plan);
    for (const auto& r : p->regions)
        if (r.name == name) { *ptr = reinterpret_cast<void*>((uintptr_t)r.base); if (bytes) *bytes = (int64_t)r.bytes; return SDK_OK; }
    return sdk_fail(SDK_ERR_ARG, "sdk_plan_region: no region named '%s'", name);
}

// host <-> named region copies and stream synchronisation, so that a plain C host needs nothing but this header
extern "C" int sdk_plan_upload(void* plan, const char* name, const void* host, int64_t bytes, void* stream) {
    void* d = nullptr; int64_t n = 0;
    const int rc = sdk_plan_region(plan, name, &d, &n);
    if (rc != SDK_OK) return rc;
    SDK_CHECK_ARG(host && bytes >= 0 && bytes <= n, "sdk_plan_upload: %lld bytes into the %lld-byte region '%s'", (long long)bytes, (long long)n, name);
    SDK_CUDA(cudaMemcpyAsync(d, host, (size_t)bytes, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
    return SDK_OK;
}
extern "C" int sdk_plan_download(void* plan, const char* name, void* host, int64_t bytes, void* stream) {
    void* d = nullptr; int64_t n = 0;
    const int rc = sdk_plan_region(plan, name, &d, &n);
    if (rc != SDK_OK) return rc;
    SDK_CHECK_ARG(host && bytes >= 0 && bytes <= n, "sdk_plan_download: %lld bytes from the %lld-byte region '%s'", (long long)bytes, (long long)n, name);
    SDK_CUDA(cudaMemcpyAsync(host, d, (size_t)bytes, cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
    return SDK_OK;
}
extern "C" int sdk_stream_create(void** stream) {
    SDK_CHECK_ARG(stream, "sdk_stream_create: null pointer");
    cudaStream_t s;
    SDK_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    *stream = s;
    return SDK_OK;
}
extern "C" int sdk_stream_sync(void* stream) { SDK_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream))); return SDK_OK; }
extern "C" int sdk_stream_destroy(void* stream) { SDK_CUDA(cudaStreamDestroy(static_cast<cudaStream_t>(stream))); return SDK_OK; }

extern "C" int sdk_plan_save(void* plan, const char* path) {
    SDK_CHECK_ARG(plan && path, "sdk_plan_save: bad arguments");
    Plan* p = static_cast<Plan*>(plan);
    const auto& reg = registry();
    for (auto& r : p->regions) r.used = !r.name.empty();                  // named (I/O) regions always travel
    // ---- encode every device pointer; anything outside the registered regions is an error (the file would not be self-contained)
    std::vector<Op> ops[MAX_PROGRAMS];
    for (int g = 0; g < MAX_PROGRAMS; ++g) {
        ops[g] = p->prog[g];
        for (size_t oi = 0; oi < ops[g].size(); ++oi) {
            Op& op = ops[g][oi];
            const FnEntry& e = reg[op.fn];
            for (int i = 0; i < op.nargs; ++i)
                if ((e.ptr_mask >> i) & 1u)
                    if (!encode_ptr(p, op.args[i], &op.args[i]))
                        return sdk_fail(SDK_ERR_ARG, "sdk_plan_save: argument %d of launch %zu of program %d (%s) points outside every registered region", i, oi, g, e.name);
            if (e.kind == FN_HANDLE || e.kind == FN_STRUCT) op.args[0] = 0;
        }
    }
    std::vector<HandleRec> hs = p->handles;
    for (size_t hi = 0; hi < hs.size(); ++hi) {
        HandleRec& h = hs[hi];
        const PtrTable t = desc_ptrs(h.kind);
        for (int i = 0; i < t.n; ++i) {
            uint64_t v;
            memcpy(&v, h.desc.data() + t.off[i], 8);
            if (!encode_ptr(p, v, &v)) return sdk_fail(SDK_ERR_ARG, "sdk_plan_save: pointer field %d of handle %zu (kind %d) points outside every registered region", i, hi, h.kind);
            memcpy(h.desc.data() + t.off[i], &v, 8);
        }
        if (h.kind == H_TC_GEMM)
            for (int i = 0; i < 2; ++i)
                if (!encode_ptr(p, h.aux[i], &h.aux[i])) return sdk_fail(SDK_ERR_ARG, "sdk_plan_save: statistics table / workspace of handle %zu points outside every registered region", hi);
    }
    std::vector<std::vector<uint8_t>> blobs = p->blobs;
    for (size_t bi = 0; bi < blobs.size(); ++bi)
        for (size_t i = 0; i < sizeof(CONV_PTRS) / sizeof(size_t); ++i) {
            uint64_t v;
            memcpy(&v, blobs[bi].data() + CONV_PTRS[i], 8);
            if (!encode_ptr(p, v, &v)) return sdk_fail(SDK_ERR_ARG, "sdk_plan_save: pointer field %zu of conv parameter block %zu points outside every registered region", i, bi);
            memcpy(blobs[bi].data() + CONV_PTRS[i], &v, 8);
        }
    FILE* f = fopen(path, "wb");
    if (!f) return sdk_fail(SDK_ERR_ARG, "sdk_plan_save: cannot open '%s' for writing", path);
    Writer w{f};
    w.raw(MAGIC, 8); w.u32(FILE_VERSION);
    w.u32((uint32_t)sizeof(SdkTcGemmDesc)); w.u32((uint32_t)sizeof(SdkAttentionTcDesc)); w.u32((uint32_t)sizeof(SdkLinearLnDesc)); w.u32((uint32_t)sizeof(SdkConvParams));
    w.u32((uint32_t)p->regions.size());
    for (const auto& r : p->regions) { w.u64(r.used ? r.bytes : 0); w.u32((uint32_t)r.kind); w.str(r.name); }
    w.u32((uint32_t)hs.size());
    for (const auto& h : hs) { w.u32((uint32_t)h.kind); w.u32((uint32_t)h.desc.size()); w.raw(h.desc.data(), h.desc.size()); w.u64(h.aux[0]); w.u64(h.aux[1]); }
    w.u32((uint32_t)blobs.size());
    for (const auto& b : blobs) { w.u32((uint32_t)b.size()); w.raw(b.data(), b.size()); }
    w.u32((uint32_t)MAX_PROGRAMS);
    for (int g = 0; g < MAX_PROGRAMS; ++g) {
        w.u32((uint32_t)ops[g].size());
        for (const Op& op : ops[g]) {
            w.str(reg[op.fn].name); w.u32((uint32_t)op.nargs);
            w.raw(op.args, sizeof(uint64_t) * op.nargs);
            w.u32((uint32_t)op.handle); w.u32((uint32_t)op.blob);
        }
    }
    // ---- contents of the constant regions (kind 0) that are referenced
    std::vector<uint8_t> host;
    for (const auto& r : p->regions) {
        if (!r.used || r.kind != 0) continue;
        host.resize(r.bytes);
        const cudaError_t e = cudaMemcpy(host.data(), reinterpret_cast<const void*>((uintptr_t)r.base), r.bytes, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { fclose(f); return sdk_fail(SDK_ERR_CUDA, "sdk_plan_save: reading region '%s': %s", r.name.c_str(), cudaGetErrorString(e)); }
        w.raw(host.data(), r.bytes);
    }
    const bool ok = w.ok;
    if (fclose(f) != 0 || !ok) return sdk_fail(SDK_ERR_ARG, "sdk_plan_save: short write to '%s'", path);
    return SDK_OK;
}

extern "C" int sdk_plan_load(const char* path, void** plan) {
    SDK_CHECK_ARG(path && plan, "sdk_plan_load: bad arguments");
    FILE* f = fopen(path, "rb");
    if (!f) return sdk_fail(SDK_ERR_ARG, "sdk_plan_load: cannot open '%s'", path);
    Reader rd{f};
    char magic[8];
    rd.raw(magic, 8);
    const uint32_t ver = rd.u32();
    const uint32_t s0 = rd.u32(), s1 = rd.u32(), s2 = rd.u32(), s3 = rd.u32();
    if (!rd.ok || memcmp(magic, MAGIC, 8) != 0 || ver != FILE_VERSION || s0 != sizeof(SdkTcGemmDesc) || s1 != sizeof(SdkAttentionTcDesc) ||
        s2 != sizeof(SdkLinearLnDesc) || s3 != sizeof(SdkConvParams)) {
        fclose(f);
        return sdk_fail(SDK_ERR_ARG, "sdk_plan_load: '%s' is not an engine file of this library version", path);
    }
    Plan* p = new (std::nothrow) Plan();
    if (!p) { fclose(f); return sdk_fail(SDK_ERR_CUDA, "out of host memory"); }
    auto bail = [&](int code, const char* what) { fclose(f); sdk_plan_destroy(p); return sdk_fail(code, "sdk_plan_load: %s ('%s')", what, path); };
    const uint32_t nreg = rd.u32();
    if (!rd.ok || nreg > (1u << 22)) return bail(SDK_ERR_ARG, "bad region table");
    uint64_t total = 0;
    std::vector<uint64_t> offs(nreg);
    for (uint32_t i = 0; i < nreg; ++i) {
        Region r;
        r.bytes = rd.u64(); r.kind = (int)rd.u32(); r.name = rd.str(); r.base = 0; r.used = r.bytes != 0;
        offs[i] = total;
        total += (r.bytes + 1023) / 1024 * 1024;              // 1 KiB alignment: TMA bases, vector loads
        p->regions.push_back(r);
    }
    if (!rd.ok) return bail(SDK_ERR_ARG, "truncated region table");
    if (total) {
        cudaError_t e = cudaMalloc(&p->slab, total);
        if (e == cudaSuccess) e = cudaMemset(p->slab, 0, total);      // scratch starts zeroed (split-K tile counters, statistics arena)
        if (e != cudaSuccess) return bail(SDK_ERR_CUDA, cudaGetErrorString(e));
    }
    std::vector<uint64_t> bases(nreg);
    for (uint32_t i = 0; i < nreg; ++i) { bases[i] = (uint64_t)(uintptr_t)p->slab + offs[i]; p->regions[i].base = p->regions[i].bytes ? bases[i] : 0; }
    const uint32_t nh = rd.u32();
    if (!rd.ok || nh > (1u << 20)) return bail(SDK_ERR_ARG, "bad handle table");
    for (uint32_t i = 0; i < nh; ++i) {
        HandleRec h;
        h.kind = (int)rd.u32(); h.h = nullptr;
        const uint32_t n = rd.u32();
        const PtrTable t = desc_ptrs(h.kind);
        if (!rd.ok || t.size == 0 || n != t.size) return bail(SDK_ERR_ARG, "bad handle record");
        h.desc.resize(n);
        rd.raw(h.desc.data(), n);
        h.aux[0] = rd.u64(); h.aux[1] = rd.u64();
        for (int k = 0; k < t.n; ++k) {
            uint64_t v;
            memcpy(&v, h.desc.data() + t.off[k], 8);
            v = decode_ptr(bases, v);
            memcpy(h.desc.data() + t.off[k], &v, 8);
        }
        if (h.kind == H_TC_GEMM) { h.aux[0] = decode_ptr(bases, h.aux[0]); h.aux[1] = decode_ptr(bases, h.aux[1]); }
        p->handles.push_back(h);
    }
    const uint32_t nb = rd.u32();
    if (!rd.ok || nb > (1u << 20)) return bail(SDK_ERR_ARG, "bad parameter-block table");
    for (uint32_t i = 0; i < nb; ++i) {
        const uint32_t n = rd.u32();
        if (!rd.ok || n != sizeof(SdkConvParams)) return bail(SDK_ERR_ARG, "bad parameter block");
        std::vector<uint8_t> b(n);
        rd.raw(b.data(), n);
        for (size_t k = 0; k < sizeof(CONV_PTRS) / sizeof(size_t); ++k) {
            uint64_t v;
            memcpy(&v, b.data() + CONV_PTRS[k], 8);
            v = decode_ptr(bases, v);
            memcpy(b.data() + CONV_PTRS[k], &v, 8);
        }
        p->blobs.push_back(b);
    }
    const uint32_t np = rd.u32();
    if (!rd.ok || np > MAX_PROGRAMS) return bail(SDK_ERR_ARG, "bad program table");
    const auto& reg = registry();
    for (uint32_t g = 0; g < np; ++g) {
        const uint32_t n = rd.u32();
        if (!rd.ok || n > (1u << 22)) return bail(SDK_ERR_ARG, "bad program");
        for (uint32_t i = 0; i < n; ++i) {
            Op op;
            memset(&op, 0, sizeof(op));
            const std::string name = rd.str();
            op.fn = find_fn(name.c_str());
            op.nargs = (int)rd.u32();
            if (!rd.ok || op.fn < 0 || op.nargs != reg[op.fn].nargs) return bail(SDK_ERR_ARG, "unknown launch in program");
            rd.raw(op.args, sizeof(uint64_t) * op.nargs);
            op.handle = (int)rd.u32(); op.blob = (int)rd.u32();
            const FnEntry& e = reg[op.fn];
            for (int k = 0; k < op.nargs; ++k) if ((e.ptr_mask >> k) & 1u) op.args[k] = decode_ptr(bases, op.args[k]);
            if ((e.kind == FN_HANDLE && (op.handle < 0 || op.handle >= (int)p->handles.size())) ||
                (e.kind == FN_STRUCT && (op.blob < 0 || op.blob >= (int)p->blobs.size()))) return bail(SDK_ERR_ARG, "launch refers to a missing handle");
            p->prog[g].push_back(op);
        }
    }
    if (!rd.ok) return bail(SDK_ERR_ARG, "truncated program table");
    // ---- constants
    std::vector<uint8_t> host;
    for (uint32_t i = 0; i < nreg; ++i) {
        const Region& r = p->regions[i];
        if (!r.bytes || r.kind != 0) continue;
        host.resize(r.bytes);
        rd.raw(host.data(), r.bytes);
        if (!rd.ok) return bail(SDK_ERR_ARG, "truncated constant data");
        const cudaError_t e = cudaMemcpy(reinterpret_cast<void*>((uintptr_t)r.base), host.data(), r.bytes, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) return bail(SDK_ERR_CUDA, cudaGetErrorString(e));
    }
    fclose(f);
    // ---- handles: TMA descriptors are encoded for the new addresses
    for (auto& h : p->handles) {
        const int rc = create_handle(h);
        if (rc != SDK_OK) { sdk_plan_destroy(p); return rc; }
    }
    *plan = p;
    return SDK_OK;
}
