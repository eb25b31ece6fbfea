// mc3_b200 -- user models compiled at run time into the fused model + chi-squared
// kernel (include/mc3b200.h, mc3b_user_model_*).
//
// The user writes `__device__ real model(real x, const real* p)`; NVRTC compiles it,
// with the kernel templates of chisq_kernel.cuh, to an sm_100a CUBIN:
//   k_model_chisq<UserModel<T, NP>, T, LC, 1, USIG>   LC = 32, 8, 1; USIG = true, false
//   k_model_eval<UserModel<T, NP>>
// A model of NX > 1 per-point inputs, `model(real x1, ..., real xNX, const real* p)`,
// becomes UserModelX<T, NP, NX> in the same kernels, with k_model_eval_x for its values.
// the same kernels, shape policy (plan_shape) and argument checks (mc3b_chisq_setup) as
// a built-in model; only the launch differs (cudaLaunchKernel on a library kernel).
// The headers NVRTC needs are embedded in the library (jit_headers.inc, written by
// build.py), so nothing reads the source tree at run time.  NVRTC itself is dlopen'ed
// from the path the caller gives: nothing links against it.
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include "chisq_args.cuh"
#include "jit_headers.inc"

namespace {

// ---- NVRTC, resolved by dlsym (the C API of nvrtc.h; result codes are ints) ----
typedef struct _nvrtcProgram* nvrtcProgram_t;
struct Nvrtc {
    int major = 0, minor = 0;
    int (*version)(int*, int*);
    const char* (*error_string)(int);
    int (*create)(nvrtcProgram_t*, const char*, const char*, int, const char* const*, const char* const*);
    int (*destroy)(nvrtcProgram_t*);
    int (*compile)(nvrtcProgram_t, int, const char* const*);
    int (*log_size)(nvrtcProgram_t, size_t*);
    int (*log)(nvrtcProgram_t, char*);
    int (*cubin_size)(nvrtcProgram_t, size_t*);
    int (*cubin)(nvrtcProgram_t, char*);
    int (*add_name)(nvrtcProgram_t, const char*);
    int (*lowered)(nvrtcProgram_t, const char*, const char**);
};

std::mutex g_nvrtc_mu;
std::map<std::string, Nvrtc> g_nvrtc;      // per path; the library stays loaded for the process

int nvrtc_open(const char* path, Nvrtc** out) {
    std::lock_guard<std::mutex> lk(g_nvrtc_mu);
    auto it = g_nvrtc.find(path);
    if (it != g_nvrtc.end()) { *out = &it->second; return MC3B_OK; }
    void* h = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    if (!h) { mc3b_set_error("cannot load NVRTC from %s: %s", path, dlerror()); return MC3B_ERR_CUDA; }
    Nvrtc n;
    bool ok = true;
    auto sym = [&](const char* name) { void* p = dlsym(h, name); ok = ok && p != nullptr; return p; };
    n.version = (int (*)(int*, int*))sym("nvrtcVersion");
    n.error_string = (const char* (*)(int))sym("nvrtcGetErrorString");
    n.create = (decltype(n.create))sym("nvrtcCreateProgram");
    n.destroy = (decltype(n.destroy))sym("nvrtcDestroyProgram");
    n.compile = (decltype(n.compile))sym("nvrtcCompileProgram");
    n.log_size = (decltype(n.log_size))sym("nvrtcGetProgramLogSize");
    n.log = (decltype(n.log))sym("nvrtcGetProgramLog");
    n.cubin_size = (decltype(n.cubin_size))sym("nvrtcGetCUBINSize");
    n.cubin = (decltype(n.cubin))sym("nvrtcGetCUBIN");
    n.add_name = (decltype(n.add_name))sym("nvrtcAddNameExpression");
    n.lowered = (decltype(n.lowered))sym("nvrtcGetLoweredName");
    if (!ok) { dlclose(h); mc3b_set_error("%s is not an NVRTC library (missing symbols)", path); return MC3B_ERR_CUDA; }
    n.version(&n.major, &n.minor);
    if (n.major * 100 + n.minor < 1208) {       // sm_100a needs NVRTC 12.8
        dlclose(h);
        mc3b_set_error("NVRTC %d.%d at %s cannot target sm_100a (needs 12.8 or newer)", n.major, n.minor, path);
        return MC3B_ERR_CUDA;
    }
    *out = &g_nvrtc.emplace(path, n).first->second;
    return MC3B_OK;
}

// The kernels of one user model: [uniform sigma][LC = 32, 8, 1], and the model values.
const int kLC[3] = {32, 8, 1};
std::string chisq_expr(int dtype, int nmodel, int ninputs, int lc, bool usig) {
    const char* t = dtype == MC3B_F64 ? "double" : "float";
    char b[160];
    if (ninputs == 1)
        snprintf(b, sizeof(b), "mc3b_jit::k_model_chisq<mc3b_jit::UserModel<%s, %d>, %s, %d, 1, %s>", t, nmodel, t,
                 lc, usig ? "true" : "false");
    else
        snprintf(b, sizeof(b), "mc3b_jit::k_model_chisq<mc3b_jit::UserModelX<%s, %d, %d>, %s, %d, 1, %s>", t, nmodel,
                 ninputs, t, lc, usig ? "true" : "false");
    return b;
}
std::string eval_expr(int dtype, int nmodel, int ninputs) {
    const char* t = dtype == MC3B_F64 ? "double" : "float";
    char b[128];
    if (ninputs == 1) snprintf(b, sizeof(b), "mc3b_jit::k_model_eval<mc3b_jit::UserModel<%s, %d>>", t, nmodel);
    else snprintf(b, sizeof(b), "mc3b_jit::k_model_eval_x<mc3b_jit::UserModelX<%s, %d, %d>>", t, nmodel, ninputs);
    return b;
}
// Their symbols (Itanium mangling of the expressions above): the CUBIN carries no
// name table, so the loader derives them; mc3b_user_model_compile checks them against
// what NVRTC lowered, so a toolchain that mangles otherwise fails at compile time.
std::string chisq_symbol(int dtype, int nmodel, int ninputs, int lc, bool usig) {
    const char t = dtype == MC3B_F64 ? 'd' : 'f';
    char b[192];
    if (ninputs == 1)
        snprintf(b, sizeof(b),
                 "_ZN8mc3b_jit13k_model_chisqINS_9UserModelI%cLi%dEEE%cLi%dELi1ELb%dEEEvN10mc3b_chisq9ChisqArgsIT0_EE",
                 t, nmodel, t, lc, usig ? 1 : 0);
    else
        snprintf(b, sizeof(b),
                 "_ZN8mc3b_jit13k_model_chisqINS_10UserModelXI%cLi%dELi%dEEE%cLi%dELi1ELb%dEEEvN10mc3b_chisq9ChisqArgsIT0_EE",
                 t, nmodel, ninputs, t, lc, usig ? 1 : 0);
    return b;
}
std::string eval_symbol(int dtype, int nmodel, int ninputs) {
    const char t = dtype == MC3B_F64 ? 'd' : 'f';
    char b[128];
    if (ninputs == 1) snprintf(b, sizeof(b), "_ZN8mc3b_jit12k_model_evalINS_9UserModelI%cLi%dEEEEEvPKdlS4_lPd", t, nmodel);
    else
        snprintf(b, sizeof(b), "_ZN8mc3b_jit14k_model_eval_xINS_10UserModelXI%cLi%dELi%dEEEEEvPKdlN10mc3b_chisq10EvalInputsElPd",
                 t, nmodel, ninputs);
    return b;
}

// What the module reports about itself (mc3b_jit_abi), checked before any launch.
enum { ABI_VERSION, ABI_ARGS_SIZE, ABI_DTYPE, ABI_NMODEL, ABI_WARPS, ABI_TILE, ABI_NINPUTS, ABI_N };

// Translation unit around the user's source; model_line: the line of `model` in it.
std::string jit_source(const char* user, int nmodel, int ninputs, int dtype, int model_line) {
    std::string s;
    s += "#include \"chisq_kernel.cuh\"\n";
    s += "namespace mc3b_user {\n";
    s += dtype == MC3B_F64 ? "typedef double real;\n" : "typedef float real;\n";
    s += "#line 1 \"model.cu\"\n";
    s += user;
    if (ninputs > 1) {
        // the call of the wrapper, reported at the line of `model`: a model of another
        // number of inputs fails to compile there
        std::string args;
        for (int j = 0; j < ninputs; j++) args += "v[" + std::to_string(j) + "], ";
        s += "\n#line " + std::to_string(model_line) + " \"model.cu\"\n";
        s += "__device__ __forceinline__ real mc3b_call_model(const real (&v)[" + std::to_string(ninputs) +
             "], const real* p) { return model(" + args + "p); }";
    }
    s += "\n}  // namespace mc3b_user\n";
    s += "#line 1 \"mc3b_jit_wrapper.cu\"\n"
         "namespace mc3b_jit {\n"
         "// the user's model behind the interface of the built-in ones (models.cuh, PolyModel)\n";
    if (ninputs == 1)
        s += "template <typename T, int NP> struct UserModel {\n"
             "    static constexpr bool GUARD = false;\n"
             "    static constexpr bool TILE_STATE = false;\n"
             "    __device__ __forceinline__ bool flagged() const { return false; }\n"
             "    __device__ __forceinline__ void clear() {}\n"
             "    T c[NP];\n"
             "    __device__ __forceinline__ void load(const double* p) {\n"
             "#pragma unroll\n"
             "        for (int k = 0; k < NP; k++) c[k] = (T)p[k];\n"
             "    }\n"
             "    __device__ __forceinline__ T eval(T x) const { return mc3b_user::model(x, c); }\n"
             "    __device__ __forceinline__ T eval_safe(T x) const { return eval(x); }\n"
             "};\n";
    else
        s += "template <typename T, int NP, int K> struct UserModelX {\n"
             "    static constexpr bool GUARD = false;\n"
             "    static constexpr bool TILE_STATE = false;\n"
             "    static constexpr int NX = K;           // per-point inputs (models.cuh ninputs_of)\n"
             "    typedef T real;\n"
             "    __device__ __forceinline__ bool flagged() const { return false; }\n"
             "    __device__ __forceinline__ void clear() {}\n"
             "    T c[NP];\n"
             "    __device__ __forceinline__ void load(const double* p) {\n"
             "#pragma unroll\n"
             "        for (int k = 0; k < NP; k++) c[k] = (T)p[k];\n"
             "    }\n"
             "    __device__ __forceinline__ T eval(const T (&v)[K]) const { return mc3b_user::mc3b_call_model(v, c); }\n"
             "    __device__ __forceinline__ T eval_safe(const T (&v)[K]) const { return eval(v); }\n"
             "};\n";
    s += "}  // namespace mc3b_jit\n";
    char b[256];
    snprintf(b, sizeof(b),
             "extern \"C\" __device__ long long mc3b_jit_abi[%d] = {MC3B_VERSION, sizeof(ChisqArgs<mc3b_user::real>), "
             "%d, %d, WARPS, tilecfg<mc3b_user::real>::TILE, %d};\n",
             (int)ABI_N, dtype, nmodel, ninputs);
    s += b;
    return s;
}

// Line (from 1) of the first `model` followed by '(' in the source, as an identifier of
// its own; 0 when there is none.
int model_line(const char* s) {
    for (const char* p = strstr(s, "model"); p; p = strstr(p + 1, "model")) {
        const char prev = p == s ? ' ' : p[-1];
        if (prev == '_' || (prev >= '0' && prev <= '9') || (prev >= 'a' && prev <= 'z') || (prev >= 'A' && prev <= 'Z'))
            continue;
        const char* q = p + 5;
        while (*q == ' ' || *q == '\t' || *q == '\n' || *q == '\r') q++;
        if (*q == '(') {
            int line = 1;
            for (const char* c = s; c < p; c++) line += *c == '\n';
            return line;
        }
    }
    return 0;
}

void copy_log(char* log, int64_t logcap, const std::string& text) {
    if (!log || logcap <= 0) return;
    const size_t n = text.size() < (size_t)(logcap - 1) ? text.size() : (size_t)(logcap - 1);
    memcpy(log, text.data(), n);
    log[n] = 0;
}

}  // namespace

struct mc3b_user_model {
    cudaLibrary_t lib;
    cudaKernel_t chisq[2][3];      // [uniform sigma][LC = 32, 8, 1]
    cudaKernel_t eval;             // k_model_eval, or k_model_eval_x for ninputs > 1
    int nmodel, ninputs, dtype;
    std::vector<char> image;       // the CUBIN, kept for the lifetime of the library
};

extern "C" int mc3b_user_model_compile_ex(const char* nvrtc_path, const char* source, int nmodel, int ninputs,
                                          int dtype, void* cubin, int64_t cap, int64_t* size, char* log,
                                          int64_t logcap) {
    MC3B_CHECK_ARG(nvrtc_path && source && size, "null pointer");
    MC3B_CHECK_ARG(nmodel >= 1 && nmodel <= MC3B_MAX_PARS, "a model takes 1 to %d parameters, got %d", MC3B_MAX_PARS,
                   nmodel);
    MC3B_CHECK_ARG(ninputs >= 1 && ninputs <= MC3B_MAX_INPUTS, "a model takes 1 to %d inputs, got %d",
                   MC3B_MAX_INPUTS, ninputs);
    MC3B_CHECK_ARG(dtype == MC3B_F64 || dtype == MC3B_F32, "bad dtype %d", dtype);
    MC3B_CHECK_ARG(cap >= 0 && (cap == 0 || cubin != nullptr), "bad CUBIN buffer");
    *size = 0;
    copy_log(log, logcap, "");
    const int line = model_line(source);
    if (line == 0) {
        const char* msg = ninputs == 1 ? "the source must define __device__ real model(real x, const real* p)"
                                       : "the source must define __device__ real model(real x1, ..., const real* p)";
        copy_log(log, logcap, msg);
        mc3b_set_error("%s", msg);
        return MC3B_ERR_ARG;
    }
    Nvrtc* nv = nullptr;
    if (int rc = nvrtc_open(nvrtc_path, &nv)) return rc;

    const std::string src = jit_source(source, nmodel, ninputs, dtype, line);
    nvrtcProgram_t prog = nullptr;
    int r = nv->create(&prog, src.c_str(), "mc3b_user_model.cu", kJitNHeaders, kJitHeaderSources, kJitHeaderNames);
    if (r != 0) { mc3b_set_error("nvrtcCreateProgram: %s", nv->error_string(r)); return MC3B_ERR_CUDA; }
    std::vector<std::string> exprs, symbols;
    for (int u = 0; u < 2; u++)
        for (int l = 0; l < 3; l++) {
            exprs.push_back(chisq_expr(dtype, nmodel, ninputs, kLC[l], u == 1));
            symbols.push_back(chisq_symbol(dtype, nmodel, ninputs, kLC[l], u == 1));
        }
    exprs.push_back(eval_expr(dtype, nmodel, ninputs));
    symbols.push_back(eval_symbol(dtype, nmodel, ninputs));
    for (const std::string& e : exprs) nv->add_name(prog, e.c_str());
    // the flags of the library's own kernels (build.py NVCC_FLAGS); -default-device: the
    // header's host prototypes (and unannotated helpers of the user) are device functions
    const char* opts[] = {"-arch=sm_100a", "-std=c++17", "--fmad=true", "-lineinfo", "-default-device"};
    r = nv->compile(prog, 5, opts);
    size_t lsz = 0;
    nv->log_size(prog, &lsz);
    std::string text(lsz, '\0');
    if (lsz > 0) nv->log(prog, &text[0]);
    while (!text.empty() && text.back() == '\0') text.pop_back();
    copy_log(log, logcap, text);
    int rc = MC3B_OK;
    if (r != 0) {
        mc3b_set_error("the user model does not compile (%s); see the log", nv->error_string(r));
        rc = MC3B_ERR_ARG;
    }
    for (size_t i = 0; rc == MC3B_OK && i < exprs.size(); i++) {
        const char* low = nullptr;
        if (nv->lowered(prog, exprs[i].c_str(), &low) != 0 || low == nullptr || symbols[i] != low) {
            mc3b_set_error("NVRTC %d.%d named %s `%s`, the loader expects `%s`", nv->major, nv->minor,
                           exprs[i].c_str(), low ? low : "(nothing)", symbols[i].c_str());
            rc = MC3B_ERR_CUDA;
        }
    }
    if (rc == MC3B_OK) {
        size_t csz = 0;
        nv->cubin_size(prog, &csz);
        *size = (int64_t)csz;
        if ((int64_t)csz > cap) {
            mc3b_set_error("the CUBIN needs %lld bytes, the buffer holds %lld", (long long)csz, (long long)cap);
            rc = MC3B_ERR_ARG;
        } else {
            nv->cubin(prog, (char*)cubin);
        }
    }
    nv->destroy(&prog);
    return rc;
}

extern "C" int mc3b_user_model_compile(const char* nvrtc_path, const char* source, int nmodel, int dtype, void* cubin,
                                       int64_t cap, int64_t* size, char* log, int64_t logcap) {
    return mc3b_user_model_compile_ex(nvrtc_path, source, nmodel, 1, dtype, cubin, cap, size, log, logcap);
}

extern "C" int mc3b_user_model_load_ex(const void* cubin, int64_t size, int nmodel, int ninputs, int dtype,
                                       mc3b_user_model_t** out) {
    MC3B_CHECK_ARG(cubin && out && size >= 64, "bad arguments");
    MC3B_CHECK_ARG(memcmp(cubin, "\x7f" "ELF", 4) == 0, "not a CUBIN (no ELF header)");
    MC3B_CHECK_ARG(nmodel >= 1 && nmodel <= MC3B_MAX_PARS, "bad nmodel %d", nmodel);
    MC3B_CHECK_ARG(ninputs >= 1 && ninputs <= MC3B_MAX_INPUTS, "bad ninputs %d", ninputs);
    MC3B_CHECK_ARG(dtype == MC3B_F64 || dtype == MC3B_F32, "bad dtype %d", dtype);
    mc3b_user_model* m = new mc3b_user_model();
    m->image.assign((const char*)cubin, (const char*)cubin + size);
    m->nmodel = nmodel;
    m->ninputs = ninputs;
    m->dtype = dtype;
    cudaError_t e = cudaLibraryLoadData(&m->lib, m->image.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) {
        delete m;
        mc3b_set_error("cudaLibraryLoadData: %s", cudaGetErrorString(e));
        return MC3B_ERR_CUDA;
    }
    auto fail = [&](int rc) { cudaLibraryUnload(m->lib); delete m; return rc; };
    // ABI guard: a module compiled against other headers (a stale disk cache) must not
    // be launched with an argument block it would misread
    void* dabi = nullptr;
    size_t bytes = 0;
    long long abi[ABI_N] = {};
    e = cudaLibraryGetGlobal(&dabi, &bytes, m->lib, "mc3b_jit_abi");
    if (e == cudaSuccess && bytes == sizeof(abi)) e = cudaMemcpy(abi, dabi, sizeof(abi), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess || bytes != sizeof(abi)) {
        mc3b_set_error("the module has no ABI record (%s)", e != cudaSuccess ? cudaGetErrorString(e) : "size");
        return fail(e != cudaSuccess ? MC3B_ERR_CUDA : MC3B_ERR_ARG);
    }
    const long long want[ABI_N] = {MC3B_VERSION,
                                   (long long)(dtype == MC3B_F64 ? sizeof(ChisqArgs<double>) : sizeof(ChisqArgs<float>)),
                                   dtype, nmodel, WARPS,
                                   dtype == MC3B_F64 ? tilecfg<double>::TILE : tilecfg<float>::TILE, ninputs};
    for (int i = 0; i < ABI_N; i++) {
        if (abi[i] != want[i]) {
            mc3b_set_error("the module does not match this library (ABI entry %d: %lld, expected %lld): "
                           "compile it again", i, abi[i], want[i]);
            return fail(MC3B_ERR_ARG);
        }
    }
    for (int u = 0; u < 2; u++)
        for (int l = 0; l < 3; l++) {
            e = cudaLibraryGetKernel(&m->chisq[u][l], m->lib,
                                     chisq_symbol(dtype, nmodel, ninputs, kLC[l], u == 1).c_str());
            if (e != cudaSuccess) { mc3b_set_error("cudaLibraryGetKernel: %s", cudaGetErrorString(e)); return fail(MC3B_ERR_CUDA); }
        }
    e = cudaLibraryGetKernel(&m->eval, m->lib, eval_symbol(dtype, nmodel, ninputs).c_str());
    if (e != cudaSuccess) { mc3b_set_error("cudaLibraryGetKernel: %s", cudaGetErrorString(e)); return fail(MC3B_ERR_CUDA); }
    *out = m;
    return MC3B_OK;
}

extern "C" int mc3b_user_model_load(const void* cubin, int64_t size, int nmodel, int dtype, mc3b_user_model_t** out) {
    return mc3b_user_model_load_ex(cubin, size, nmodel, 1, dtype, out);
}

extern "C" int mc3b_user_model_free(mc3b_user_model_t* m) {
    if (m == nullptr) return MC3B_OK;
    const cudaError_t e = cudaLibraryUnload(m->lib);
    delete m;
    MC3B_CUDA(e);
    return MC3B_OK;
}

namespace {
template <typename T>
int user_chisq_t(const mc3b_user_model_t* m, const double* params, int64_t ldp, int64_t nchains,
                 const void* const* xs, const void* d, const void* w, int64_t n, double* partial, int64_t ldpartial,
                 int nsplit, const mc3b_chisq_opts_t& o, cudaStream_t st) {
    ChisqArgs<T> A;
    Shape sh;
    dim3 grid;
    const int rc = mc3b_chisq_setup<T>(params, ldp, nchains, xs[0], d, w, n, partial, ldpartial, nsplit, m->dtype, o,
                                       A, sh, grid);
    if (rc != MC3B_OK) return rc;
    for (int j = 1; j < m->ninputs; j++) {
        A.xs[j] = (const T*)xs[j];
        if (((uintptr_t)xs[j] & 15) != 0) A.use_tma = 0;     // TMA needs 16-byte aligned tiles
    }
    const int u = o.uniform_sigma != 0 ? 1 : 0;
    const int l = sh.lc == 32 ? 0 : (sh.lc == 8 ? 1 : 2);
    void* args[] = {&A};
    MC3B_CUDA(cudaLaunchKernel((const void*)m->chisq[u][l], grid, dim3(WARPS * 32), args, 0, st));
    return MC3B_OK;
}

int user_chisq(const mc3b_user_model_t* m, const double* params, int64_t ldp, int64_t nchains, const void* const* xs,
               const void* data, const void* invsig, int64_t n, double* partial, int64_t ldpartial, int nsplit,
               const mc3b_chisq_opts_t* opts, void* stream) {
    MC3B_CHECK_ARG(params && data && invsig && partial, "null pointer");
    for (int j = 0; j < m->ninputs; j++) MC3B_CHECK_ARG(xs[j], "null pointer (input %d)", j);
    MC3B_CHECK_ARG(ldpartial >= nchains, "ldpartial < nchains");
    MC3B_CHECK_ARG(nchains > 0 && n > 0 && m->nmodel <= ldp, "bad sizes");
    mc3b_chisq_opts_t o = {};
    if (opts) o = *opts;
    MC3B_CHECK_ARG(!o.folded && !o.work && !o.moment && !o.tile_x,
                   "user models take plan_chains, uniform_sigma and the fuse options only "
                   "(folded, work, moment and tile_x belong to the grid sinusoid)");
    cudaStream_t st = (cudaStream_t)stream;
    if (m->dtype == MC3B_F64)
        return user_chisq_t<double>(m, params, ldp, nchains, xs, data, invsig, n, partial, ldpartial, nsplit, o, st);
    return user_chisq_t<float>(m, params, ldp, nchains, xs, data, invsig, n, partial, ldpartial, nsplit, o, st);
}

int user_eval(const mc3b_user_model_t* m, const double* params, int64_t ldp, int64_t nchains,
              const double* const* xs, int64_t n, double* out, void* stream) {
    MC3B_CHECK_ARG(params && out && nchains > 0 && n > 0 && m->nmodel <= ldp, "bad arguments");
    for (int j = 0; j < m->ninputs; j++) MC3B_CHECK_ARG(xs[j], "null pointer (input %d)", j);
    MC3B_CHECK_ARG(nchains <= 65535, "model_eval is for small batches (<= 65535 rows)");
    int64_t bx = ceil_div64(n, 256);
    if (bx > 1184) bx = 1184;
    EvalInputs in = {};
    for (int j = 0; j < m->ninputs; j++) in.x[j] = xs[j];
    void* args1[] = {&params, &ldp, &in.x[0], &n, &out};
    void* argsx[] = {&params, &ldp, &in, &n, &out};
    MC3B_CUDA(cudaLaunchKernel((const void*)m->eval, dim3((unsigned)bx, (unsigned)nchains), dim3(256),
                               m->ninputs == 1 ? args1 : argsx, 0, (cudaStream_t)stream));
    return MC3B_OK;
}
}  // namespace

extern "C" int mc3b_user_model_chisq_ex(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                        int64_t nchains, const void* x, const void* data, const void* invsig,
                                        int64_t n, double* partial, int64_t ldpartial, int nsplit,
                                        const mc3b_chisq_opts_t* opts, void* stream) {
    MC3B_CHECK_ARG(m && x, "null pointer");
    MC3B_CHECK_ARG(m->ninputs == 1, "this model takes %d inputs: launch it with mc3b_user_model_chisq_inputs",
                   m->ninputs);
    return user_chisq(m, params, ldp, nchains, &x, data, invsig, n, partial, ldpartial, nsplit, opts, stream);
}

extern "C" int mc3b_user_model_chisq_inputs(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                            int64_t nchains, const void* const* xs, int nx, const void* data,
                                            const void* invsig, int64_t n, double* partial, int64_t ldpartial,
                                            int nsplit, const mc3b_chisq_opts_t* opts, void* stream) {
    MC3B_CHECK_ARG(m && xs, "null pointer");
    MC3B_CHECK_ARG(nx == m->ninputs, "this model takes %d inputs, got %d", m->ninputs, nx);
    return user_chisq(m, params, ldp, nchains, xs, data, invsig, n, partial, ldpartial, nsplit, opts, stream);
}

extern "C" int mc3b_user_model_eval(const mc3b_user_model_t* m, const double* params, int64_t ldp, int64_t nchains,
                                    const double* x, int64_t n, double* out, void* stream) {
    MC3B_CHECK_ARG(m && x, "bad arguments");
    MC3B_CHECK_ARG(m->ninputs == 1, "this model takes %d inputs: evaluate it with mc3b_user_model_eval_inputs",
                   m->ninputs);
    return user_eval(m, params, ldp, nchains, &x, n, out, stream);
}

extern "C" int mc3b_user_model_eval_inputs(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                           int64_t nchains, const double* const* xs, int nx, int64_t n, double* out,
                                           void* stream) {
    MC3B_CHECK_ARG(m && xs, "bad arguments");
    MC3B_CHECK_ARG(nx == m->ninputs, "this model takes %d inputs, got %d", m->ninputs, nx);
    return user_eval(m, params, ldp, nchains, xs, n, out, stream);
}
