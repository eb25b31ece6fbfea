// mc3_b200 -- user models compiled at run time into the fused model + chi-squared
// kernel (include/mc3b200.h, mc3b_user_model_*).
//
// The user writes `__device__ real model(real x, const real* p)`; NVRTC compiles it,
// with the kernel templates of chisq_kernel.cuh, to an sm_100a CUBIN:
//   k_model_chisq<UserModel<T, NP>, T, LC, 1, USIG>   LC = 32, 8, 1; USIG = true, false
//   k_model_eval<UserModel<T, NP>>
// A model of NX > 1 per-point inputs, `model(real x1, ..., real xNX, const real* p)`,
// becomes UserModelX<T, NP, NX> in the same kernels, with k_model_eval_x for its values.
// A model of run-time constants, work slots or a `prepare(real* p)` step becomes
// UserModelK<T, NP, NX, NC, NW> (p = [parameters | constants | work], prepare run in load),
// with k_model_eval_k; whether the source defines prepare is asked of NVRTC first, by a
// small probe compile (prepare_probe).  A user model runs in
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
#include "dwt_kernel.cuh"
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
// A model of run-time constants, work slots or a prepare step (d.kind) is a
// UserModelK<T, NP, NX, NC, NW>, with k_model_eval_k for its values; any other keeps the
// UserModel / UserModelX names it had before models took constants.
const int kLC[3] = {32, 8, 1};
struct Desc {
    int nmodel, ninputs, nconst, nwork, dtype;
    bool prepare;                  // the source defines prepare (prepare_probe)
    bool k() const { return nconst > 0 || nwork > 0 || prepare; }
};
std::string wrapper_expr(const Desc& d) {
    const char* t = d.dtype == MC3B_F64 ? "double" : "float";
    char b[96];
    if (d.k())
        snprintf(b, sizeof(b), "mc3b_jit::UserModelK<%s, %d, %d, %d, %d>", t, d.nmodel, d.ninputs, d.nconst, d.nwork);
    else if (d.ninputs == 1) snprintf(b, sizeof(b), "mc3b_jit::UserModel<%s, %d>", t, d.nmodel);
    else snprintf(b, sizeof(b), "mc3b_jit::UserModelX<%s, %d, %d>", t, d.nmodel, d.ninputs);
    return b;
}
std::string chisq_expr(const Desc& d, int lc, bool usig) {
    const char* t = d.dtype == MC3B_F64 ? "double" : "float";
    char b[224];
    snprintf(b, sizeof(b), "mc3b_jit::k_model_chisq<%s, %s, %d, 1, %s>", wrapper_expr(d).c_str(), t, lc,
             usig ? "true" : "false");
    return b;
}
std::string eval_expr(const Desc& d) {
    const char* k = d.k() ? "k_model_eval_k" : d.ninputs == 1 ? "k_model_eval" : "k_model_eval_x";
    return std::string("mc3b_jit::") + k + "<" + wrapper_expr(d) + ">";
}
// Their symbols (Itanium mangling of the expressions above): the CUBIN carries no
// name table, so the loader derives them; mc3b_user_model_compile checks them against
// what NVRTC lowered, so a toolchain that mangles otherwise fails at compile time.
std::string wrapper_symbol(const Desc& d) {
    const char t = d.dtype == MC3B_F64 ? 'd' : 'f';
    char b[96];
    if (d.k())
        snprintf(b, sizeof(b), "10UserModelKI%cLi%dELi%dELi%dELi%dEE", t, d.nmodel, d.ninputs, d.nconst, d.nwork);
    else if (d.ninputs == 1) snprintf(b, sizeof(b), "9UserModelI%cLi%dEE", t, d.nmodel);
    else snprintf(b, sizeof(b), "10UserModelXI%cLi%dELi%dEE", t, d.nmodel, d.ninputs);
    return b;
}
std::string chisq_symbol(const Desc& d, int lc, bool usig) {
    const char t = d.dtype == MC3B_F64 ? 'd' : 'f';
    char b[224];
    snprintf(b, sizeof(b), "_ZN8mc3b_jit13k_model_chisqINS_%sE%cLi%dELi1ELb%dEEEvN10mc3b_chisq9ChisqArgsIT0_EE",
             wrapper_symbol(d).c_str(), t, lc, usig ? 1 : 0);
    return b;
}
std::string eval_symbol(const Desc& d) {
    const std::string w = wrapper_symbol(d);
    if (d.k()) return "_ZN8mc3b_jit14k_model_eval_kINS_" + w + "EEEvPKdlN10mc3b_chisq10EvalInputsES4_lPd";
    if (d.ninputs == 1) return "_ZN8mc3b_jit12k_model_evalINS_" + w + "EEEvPKdlS4_lPd";
    return "_ZN8mc3b_jit14k_model_eval_xINS_" + w + "EEEvPKdlN10mc3b_chisq10EvalInputsElPd";
}

// The D4 kernels of an fp64 module that read the model (dwt_kernel.cuh): the wavelet
// likelihood's first pass.  [0] k_dwt_reg_model, [1] k_dwt_pass<SRC_MODEL>, [2] k_dwt_last<SRC_MODEL>
std::string dwt_expr(const Desc& d, int k) {
    const std::string w = wrapper_expr(d);
    if (k == 0) return "mc3b_jit::k_dwt_reg_model<" + w + ", mc3b_jit::RegArgsX>";
    if (k == 1) return "mc3b_jit::k_dwt_pass<mc3b_jit::SRC_MODEL, " + w + ", mc3b_jit::PassArgsX>";
    return "mc3b_jit::k_dwt_last<mc3b_jit::SRC_MODEL, " + w + ", mc3b_jit::LastArgsX>";
}
std::string dwt_symbol(const Desc& d, int k) {
    const std::string w = wrapper_symbol(d);
    if (k == 0) return "_ZN8mc3b_jit15k_dwt_reg_modelINS_" + w + "ENS_8RegArgsXEEEvT0_";
    if (k == 1) return "_ZN8mc3b_jit10k_dwt_passILi0ENS_" + w + "ENS_9PassArgsXEEEvT1_";
    return "_ZN8mc3b_jit10k_dwt_lastILi0ENS_" + w + "ENS_9LastArgsXEEEvT1_";
}
// sizes of the three argument blocks, one entry of the ABI record
constexpr long long kDwtArgsSizes =
    (long long)sizeof(RegArgsX) | (long long)sizeof(PassArgsX) << 16 | (long long)sizeof(LastArgsX) << 32;

// What the module reports about itself (mc3b_jit_abi), checked before any launch.
enum { ABI_VERSION, ABI_ARGS_SIZE, ABI_DTYPE, ABI_NMODEL, ABI_WARPS, ABI_TILE, ABI_NINPUTS, ABI_NCONST, ABI_NWORK,
       ABI_PREPARE, ABI_DWT_ARGS, ABI_N };

// The user's source in its namespace, with `real` defined and line numbers of model.cu.
std::string user_unit(const char* user, int dtype) {
    std::string s;
    s += "#include \"chisq_kernel.cuh\"\n";
    s += "namespace mc3b_user {\n";
    s += dtype == MC3B_F64 ? "typedef double real;\n" : "typedef float real;\n";
    s += "#line 1 \"model.cu\"\n";
    s += user;
    return s;
}

// Translation unit around the user's source; model_line / prepare_line: the lines of
// `model` and `prepare` in it.
std::string jit_source(const char* user, const Desc& d, int model_line, int prepare_line) {
    std::string s = "#include \"dwt_kernel.cuh\"\n" + user_unit(user, d.dtype);
    const int ninputs = d.ninputs;
    if (ninputs > 1) {
        // the call of the wrapper, reported at the line of `model`: a model of another
        // number of inputs fails to compile there
        std::string args;
        for (int j = 0; j < ninputs; j++) args += "v[" + std::to_string(j) + "], ";
        s += "\n#line " + std::to_string(model_line) + " \"model.cu\"\n";
        s += "__device__ __forceinline__ real mc3b_call_model(const real (&v)[" + std::to_string(ninputs) +
             "], const real* p) { return model(" + args + "p); }";
    }
    if (d.prepare) {
        s += "\n#line " + std::to_string(prepare_line) + " \"model.cu\"\n";
        s += "__device__ __forceinline__ void mc3b_call_prepare(real* p) { prepare(p); }";
    }
    s += "\n}  // namespace mc3b_user\n";
    s += "#line 1 \"mc3b_jit_wrapper.cu\"\n"
         "namespace mc3b_jit {\n"
         "// the user's model behind the interface of the built-in ones (models.cuh, PolyModel)\n";
    if (d.k()) {
        s += "template <typename T, int NP, int K, int NCONST, int NWORK> struct UserModelK {\n"
             "    static constexpr bool GUARD = false;\n"
             "    static constexpr bool TILE_STATE = false;\n"
             "    static constexpr int NX = K;           // per-point inputs (models.cuh ninputs_of)\n"
             "    static constexpr int NC = NCONST;      // load(p, k) (models.cuh takes_consts)\n"
             "    typedef T real;\n"
             "    __device__ __forceinline__ bool flagged() const { return false; }\n"
             "    __device__ __forceinline__ void clear() {}\n"
             "    T c[NP + NCONST + NWORK];              // [parameters | constants | work]\n"
             "    template <typename C> __device__ __forceinline__ void load(const double* p, const C* k) {\n"
             "#pragma unroll\n"
             "        for (int j = 0; j < NP; j++) c[j] = (T)p[j];\n"
             "#pragma unroll\n"
             "        for (int j = 0; j < NCONST; j++) c[NP + j] = (T)k[j];\n"
             "#pragma unroll\n"
             "        for (int j = 0; j < NWORK; j++) c[NP + NCONST + j] = (T)0;\n";
        if (d.prepare) s += "        mc3b_user::mc3b_call_prepare(c);\n";
        s += "    }\n";
        if (ninputs == 1)
            s += "    __device__ __forceinline__ T eval(T x) const { return mc3b_user::model(x, c); }\n"
                 "    __device__ __forceinline__ T eval_safe(T x) const { return eval(x); }\n";
        else
            s += "    __device__ __forceinline__ T eval(const T (&v)[K]) const { return mc3b_user::mc3b_call_model(v, c); }\n"
                 "    __device__ __forceinline__ T eval_safe(const T (&v)[K]) const { return eval(v); }\n";
        s += "};\n";
    } else if (ninputs == 1) {
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
    } else {
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
    }
    s += "}  // namespace mc3b_jit\n";
    char b[480];
    snprintf(b, sizeof(b),
             "extern \"C\" __device__ long long mc3b_jit_abi[%d] = {MC3B_VERSION, sizeof(ChisqArgs<mc3b_user::real>), "
             "%d, %d, WARPS, tilecfg<mc3b_user::real>::TILE, %d, %d, %d, %d, (long long)sizeof(mc3b_jit::RegArgsX) | "
             "(long long)sizeof(mc3b_jit::PassArgsX) << 16 | (long long)sizeof(mc3b_jit::LastArgsX) << 32};\n",
             (int)ABI_N, d.dtype, d.nmodel, ninputs, d.nconst, d.nwork, d.prepare ? 1 : 0);
    s += b;
    return s;
}

// Translation unit that asks whether the user's source defines `prepare`: unqualified
// lookup from inside mc3b_user finds the user's own `prepare` when there is one (it hides
// the global fallback), and the fallback otherwise.  The answer is the template argument
// of mc3b_prepare_probe, read back from its lowered name.  A `prepare` that cannot take a
// real* makes the decltype fail, reported at prepare_line of model.cu.
std::string probe_source(const char* user, int dtype, int prepare_line) {
    std::string s =
        "struct mc3b_no_prepare {};\n"
        "template <class P> __device__ mc3b_no_prepare prepare(P) { return mc3b_no_prepare(); }\n"
        "template <class A, class B> struct mc3b_same { static constexpr bool value = false; };\n"
        "template <class A> struct mc3b_same<A, A> { static constexpr bool value = true; };\n"
        "template <bool B> __global__ void mc3b_prepare_probe() {}\n";
    s += user_unit(user, dtype);
    s += "\n#line " + std::to_string(prepare_line) + " \"model.cu\"\n";
    s += "constexpr bool mc3b_has_prepare = !mc3b_same<decltype(prepare((real*)nullptr)), ::mc3b_no_prepare>::value;\n";
    s += "}  // namespace mc3b_user\n";
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

// Line of the first identifier `name` outside comments and literals; 1 when there is
// none.  Only where errors are reported depends on it: whether `prepare` exists is asked
// of the compiler (probe_source).
int code_line(const char* s, const char* name) {
    const size_t len = strlen(name);
    auto ident = [](char c) { return c == '_' || (c >= '0' && c <= '9') || (c >= 'a' && c <= 'z') || (c >= 'A' && c <= 'Z'); };
    int line = 1;
    for (const char* p = s; *p; p++) {
        if (p[0] == '/' && p[1] == '/') {
            while (*p && *p != '\n') p++;
            if (!*p) break;
        } else if (p[0] == '/' && p[1] == '*') {
            for (p += 2; *p && !(p[0] == '*' && p[1] == '/'); p++) line += *p == '\n';
            if (!*p) break;
            p++;
            continue;
        } else if (*p == '"' || *p == '\'') {
            const char q = *p;
            for (p++; *p && *p != q && *p != '\n'; p++)
                if (*p == '\\' && p[1]) p++;
            if (!*p) break;
            if (*p != '\n') continue;
        } else if (strncmp(p, name, len) == 0 && (p == s || !ident(p[-1])) && !ident(p[len])) {
            return line;
        }
        line += *p == '\n';
    }
    return 1;
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
    cudaKernel_t eval;             // k_model_eval, k_model_eval_x (ninputs > 1) or k_model_eval_k (Desc::k)
    cudaKernel_t dwt[3];           // fp64: dwt_expr's kernels; fp32: none
    Desc d;
    std::vector<char> image;       // the CUBIN, kept for the lifetime of the library
};

namespace {
// NVRTC log of prog, into text and the caller's buffer
std::string program_log(Nvrtc* nv, nvrtcProgram_t prog, char* log, int64_t logcap) {
    size_t lsz = 0;
    nv->log_size(prog, &lsz);
    std::string text(lsz, '\0');
    if (lsz > 0) nv->log(prog, &text[0]);
    while (!text.empty() && text.back() == '\0') text.pop_back();
    copy_log(log, logcap, text);
    return text;
}

// the flags of the library's own kernels (build.py NVCC_FLAGS); -default-device: the
// header's host prototypes (and unannotated helpers of the user) are device functions
const char* const kOpts[] = {"-arch=sm_100a", "-std=c++17", "--fmad=true", "-lineinfo", "-default-device"};

// Does the source define prepare?  (probe_source)  MC3B_ERR_ARG with the log when the
// source does not compile.
int prepare_probe(Nvrtc* nv, const char* source, int dtype, int prepare_line, bool* found, char* log,
                  int64_t logcap) {
    const std::string src = probe_source(source, dtype, prepare_line);
    nvrtcProgram_t prog = nullptr;
    int r = nv->create(&prog, src.c_str(), "mc3b_user_model.cu", kJitNHeaders, kJitHeaderSources, kJitHeaderNames);
    if (r != 0) { mc3b_set_error("nvrtcCreateProgram: %s", nv->error_string(r)); return MC3B_ERR_CUDA; }
    const char* expr = "mc3b_prepare_probe<mc3b_user::mc3b_has_prepare>";
    nv->add_name(prog, expr);
    r = nv->compile(prog, 5, kOpts);
    program_log(nv, prog, log, logcap);
    int rc = MC3B_OK;
    const char* low = nullptr;
    if (r != 0) {
        mc3b_set_error("the user model does not compile (%s); see the log", nv->error_string(r));
        rc = MC3B_ERR_ARG;
    } else if (nv->lowered(prog, expr, &low) != 0 || low == nullptr ||
               (strcmp(low, "_Z18mc3b_prepare_probeILb0EEvv") != 0 && strcmp(low, "_Z18mc3b_prepare_probeILb1EEvv") != 0)) {
        mc3b_set_error("NVRTC %d.%d named %s `%s`", nv->major, nv->minor, expr, low ? low : "(nothing)");
        rc = MC3B_ERR_CUDA;
    } else {
        *found = strcmp(low, "_Z18mc3b_prepare_probeILb1EEvv") == 0;
    }
    nv->destroy(&prog);
    return rc;
}

int check_desc(const mc3b_user_model_desc_t* d) {
    MC3B_CHECK_ARG(d != nullptr, "null pointer");
    MC3B_CHECK_ARG(d->nmodel >= 1 && d->nmodel <= MC3B_MAX_PARS, "a model takes 1 to %d parameters, got %d",
                   MC3B_MAX_PARS, d->nmodel);
    MC3B_CHECK_ARG(d->ninputs >= 1 && d->ninputs <= MC3B_MAX_INPUTS, "a model takes 1 to %d inputs, got %d",
                   MC3B_MAX_INPUTS, d->ninputs);
    MC3B_CHECK_ARG(d->nconst >= 0 && d->nwork >= 0, "nconst and nwork must not be negative (got %d, %d)",
                   d->nconst, d->nwork);
    MC3B_CHECK_ARG(d->nmodel + d->nconst + d->nwork <= MC3B_MAX_PARS,
                   "nparams + nconst + nwork = %d + %d + %d exceeds the %d slots of a model", d->nmodel, d->nconst,
                   d->nwork, MC3B_MAX_PARS);
    MC3B_CHECK_ARG(d->dtype == MC3B_F64 || d->dtype == MC3B_F32, "bad dtype %d", d->dtype);
    return MC3B_OK;
}
}  // namespace

extern "C" int mc3b_user_model_compile_desc(const char* nvrtc_path, const char* source,
                                            const mc3b_user_model_desc_t* desc, void* cubin, int64_t cap,
                                            int64_t* size, char* log, int64_t logcap) {
    MC3B_CHECK_ARG(nvrtc_path && source && size, "null pointer");
    if (int rc = check_desc(desc)) return rc;
    MC3B_CHECK_ARG(cap >= 0 && (cap == 0 || cubin != nullptr), "bad CUBIN buffer");
    Desc d = {desc->nmodel, desc->ninputs, desc->nconst, desc->nwork, desc->dtype, false};
    *size = 0;
    copy_log(log, logcap, "");
    const int line = model_line(source);
    if (line == 0) {
        const char* msg = d.ninputs == 1 ? "the source must define __device__ real model(real x, const real* p)"
                                         : "the source must define __device__ real model(real x1, ..., const real* p)";
        copy_log(log, logcap, msg);
        mc3b_set_error("%s", msg);
        return MC3B_ERR_ARG;
    }
    Nvrtc* nv = nullptr;
    if (int rc = nvrtc_open(nvrtc_path, &nv)) return rc;
    const int pline = code_line(source, "prepare");
    if (int rc = prepare_probe(nv, source, d.dtype, pline, &d.prepare, log, logcap)) return rc;
    if (d.nwork > 0 && !d.prepare) {
        char msg[160];
        snprintf(msg, sizeof(msg), "nwork = %d work slots need __device__ void prepare(real* p) to fill them; "
                 "the source defines no prepare", d.nwork);
        copy_log(log, logcap, msg);
        mc3b_set_error("%s", msg);
        return MC3B_ERR_ARG;
    }

    const std::string src = jit_source(source, d, line, pline);
    nvrtcProgram_t prog = nullptr;
    int r = nv->create(&prog, src.c_str(), "mc3b_user_model.cu", kJitNHeaders, kJitHeaderSources, kJitHeaderNames);
    if (r != 0) { mc3b_set_error("nvrtcCreateProgram: %s", nv->error_string(r)); return MC3B_ERR_CUDA; }
    std::vector<std::string> exprs, symbols;
    for (int u = 0; u < 2; u++)
        for (int l = 0; l < 3; l++) {
            exprs.push_back(chisq_expr(d, kLC[l], u == 1));
            symbols.push_back(chisq_symbol(d, kLC[l], u == 1));
        }
    exprs.push_back(eval_expr(d));
    symbols.push_back(eval_symbol(d));
    for (int k = 0; d.dtype == MC3B_F64 && k < 3; k++) {
        exprs.push_back(dwt_expr(d, k));
        symbols.push_back(dwt_symbol(d, k));
    }
    for (const std::string& e : exprs) nv->add_name(prog, e.c_str());
    r = nv->compile(prog, 5, kOpts);
    program_log(nv, prog, log, logcap);
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

extern "C" int mc3b_user_model_compile_ex(const char* nvrtc_path, const char* source, int nmodel, int ninputs,
                                          int dtype, void* cubin, int64_t cap, int64_t* size, char* log,
                                          int64_t logcap) {
    const mc3b_user_model_desc_t d = {nmodel, ninputs, 0, 0, dtype};
    return mc3b_user_model_compile_desc(nvrtc_path, source, &d, cubin, cap, size, log, logcap);
}

extern "C" int mc3b_user_model_compile(const char* nvrtc_path, const char* source, int nmodel, int dtype, void* cubin,
                                       int64_t cap, int64_t* size, char* log, int64_t logcap) {
    return mc3b_user_model_compile_ex(nvrtc_path, source, nmodel, 1, dtype, cubin, cap, size, log, logcap);
}

extern "C" int mc3b_user_model_load_desc(const void* cubin, int64_t size, const mc3b_user_model_desc_t* desc,
                                         mc3b_user_model_t** out) {
    MC3B_CHECK_ARG(cubin && out && size >= 64, "bad arguments");
    MC3B_CHECK_ARG(memcmp(cubin, "\x7f" "ELF", 4) == 0, "not a CUBIN (no ELF header)");
    if (int rc = check_desc(desc)) return rc;
    mc3b_user_model* m = new mc3b_user_model();
    m->image.assign((const char*)cubin, (const char*)cubin + size);
    m->d = Desc{desc->nmodel, desc->ninputs, desc->nconst, desc->nwork, desc->dtype, false};
    const int dtype = desc->dtype;
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
    // whether the source defines prepare is the module's to say (entry ABI_PREPARE)
    const long long want[ABI_N] = {MC3B_VERSION,
                                   (long long)(dtype == MC3B_F64 ? sizeof(ChisqArgs<double>) : sizeof(ChisqArgs<float>)),
                                   dtype, desc->nmodel, WARPS,
                                   dtype == MC3B_F64 ? tilecfg<double>::TILE : tilecfg<float>::TILE, desc->ninputs,
                                   desc->nconst, desc->nwork, abi[ABI_PREPARE] == 1 || desc->nwork > 0 ? 1 : 0,
                                   kDwtArgsSizes};
    for (int i = 0; i < ABI_N; i++) {
        if (abi[i] != want[i]) {
            mc3b_set_error("the module does not match this library (ABI entry %d: %lld, expected %lld): "
                           "compile it again", i, abi[i], want[i]);
            return fail(MC3B_ERR_ARG);
        }
    }
    m->d.prepare = abi[ABI_PREPARE] == 1;
    for (int u = 0; u < 2; u++)
        for (int l = 0; l < 3; l++) {
            e = cudaLibraryGetKernel(&m->chisq[u][l], m->lib, chisq_symbol(m->d, kLC[l], u == 1).c_str());
            if (e != cudaSuccess) { mc3b_set_error("cudaLibraryGetKernel: %s", cudaGetErrorString(e)); return fail(MC3B_ERR_CUDA); }
        }
    e = cudaLibraryGetKernel(&m->eval, m->lib, eval_symbol(m->d).c_str());
    if (e != cudaSuccess) { mc3b_set_error("cudaLibraryGetKernel: %s", cudaGetErrorString(e)); return fail(MC3B_ERR_CUDA); }
    if (dtype == MC3B_F64) {
        for (int k = 0; k < 3; k++) {
            e = cudaLibraryGetKernel(&m->dwt[k], m->lib, dwt_symbol(m->d, k).c_str());
            if (e != cudaSuccess) { mc3b_set_error("cudaLibraryGetKernel: %s", cudaGetErrorString(e)); return fail(MC3B_ERR_CUDA); }
        }
        // k_dwt_pass takes more than 48 KB of dynamic shared memory: set here, once per device,
        // so that no launch (or graph capture) has to
        int ndev = 0;
        e = cudaGetDeviceCount(&ndev);
        for (int dev = 0; e == cudaSuccess && dev < ndev; dev++)
            e = cudaKernelSetAttributeForDevice(m->dwt[1], cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                (int)pass_smem(m->d.ninputs), dev);
        if (e != cudaSuccess) { mc3b_set_error("k_dwt_pass shared memory: %s", cudaGetErrorString(e)); return fail(MC3B_ERR_CUDA); }
    }
    *out = m;
    return MC3B_OK;
}

extern "C" int mc3b_user_model_load_ex(const void* cubin, int64_t size, int nmodel, int ninputs, int dtype,
                                       mc3b_user_model_t** out) {
    const mc3b_user_model_desc_t d = {nmodel, ninputs, 0, 0, dtype};
    return mc3b_user_model_load_desc(cubin, size, &d, out);
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
                 const void* const* xs, const void* consts, const void* d, const void* w, int64_t n, double* partial,
                 int64_t ldpartial, int nsplit, const mc3b_chisq_opts_t& o, cudaStream_t st) {
    ChisqArgs<T> A;
    Shape sh;
    dim3 grid;
    const int rc = mc3b_chisq_setup<T>(params, ldp, nchains, xs[0], d, w, n, partial, ldpartial, nsplit, m->d.dtype, o,
                                       A, sh, grid);
    if (rc != MC3B_OK) return rc;
    for (int j = 1; j < m->d.ninputs; j++) {
        A.xs[j] = (const T*)xs[j];
        if (((uintptr_t)xs[j] & 15) != 0) A.use_tma = 0;     // TMA needs 16-byte aligned tiles
    }
    A.uconst = (const T*)consts;
    const int u = o.uniform_sigma != 0 ? 1 : 0;
    const int l = sh.lc == 32 ? 0 : (sh.lc == 8 ? 1 : 2);
    void* args[] = {&A};
    MC3B_CUDA(cudaLaunchKernel((const void*)m->chisq[u][l], grid, dim3(WARPS * 32), args, 0, st));
    return MC3B_OK;
}

int user_chisq(const mc3b_user_model_t* m, const double* params, int64_t ldp, int64_t nchains, const void* const* xs,
               const void* consts, const void* data, const void* invsig, int64_t n, double* partial,
               int64_t ldpartial, int nsplit, const mc3b_chisq_opts_t* opts, void* stream) {
    MC3B_CHECK_ARG(params && data && invsig && partial, "null pointer");
    for (int j = 0; j < m->d.ninputs; j++) MC3B_CHECK_ARG(xs[j], "null pointer (input %d)", j);
    MC3B_CHECK_ARG(consts || m->d.nconst == 0, "null pointer (constants)");
    MC3B_CHECK_ARG(ldpartial >= nchains, "ldpartial < nchains");
    MC3B_CHECK_ARG(nchains > 0 && n > 0 && m->d.nmodel <= ldp, "bad sizes");
    mc3b_chisq_opts_t o = {};
    if (opts) o = *opts;
    MC3B_CHECK_ARG(!o.folded && !o.work && !o.moment && !o.tile_x,
                   "user models take plan_chains, uniform_sigma and the fuse options only "
                   "(folded, work, moment and tile_x belong to the grid sinusoid)");
    cudaStream_t st = (cudaStream_t)stream;
    if (m->d.dtype == MC3B_F64)
        return user_chisq_t<double>(m, params, ldp, nchains, xs, consts, data, invsig, n, partial, ldpartial, nsplit,
                                    o, st);
    return user_chisq_t<float>(m, params, ldp, nchains, xs, consts, data, invsig, n, partial, ldpartial, nsplit, o,
                               st);
}

int user_eval(const mc3b_user_model_t* m, const double* params, int64_t ldp, int64_t nchains,
              const double* const* xs, const double* consts, int64_t n, double* out, void* stream) {
    MC3B_CHECK_ARG(params && out && nchains > 0 && n > 0 && m->d.nmodel <= ldp, "bad arguments");
    for (int j = 0; j < m->d.ninputs; j++) MC3B_CHECK_ARG(xs[j], "null pointer (input %d)", j);
    MC3B_CHECK_ARG(consts || m->d.nconst == 0, "null pointer (constants)");
    MC3B_CHECK_ARG(nchains <= 65535, "model_eval is for small batches (<= 65535 rows)");
    int64_t bx = ceil_div64(n, 256);
    if (bx > 1184) bx = 1184;
    EvalInputs in = {};
    for (int j = 0; j < m->d.ninputs; j++) in.x[j] = xs[j];
    void* args1[] = {&params, &ldp, &in.x[0], &n, &out};
    void* argsx[] = {&params, &ldp, &in, &n, &out};
    void* argsk[] = {&params, &ldp, &in, &consts, &n, &out};
    MC3B_CUDA(cudaLaunchKernel((const void*)m->eval, dim3((unsigned)bx, (unsigned)nchains), dim3(256),
                               m->d.k() ? argsk : m->d.ninputs == 1 ? args1 : argsx, 0, (cudaStream_t)stream));
    return MC3B_OK;
}
}  // namespace

#define MC3B_NO_CONSTS(m, entry)                                                                   \
    MC3B_CHECK_ARG((m)->d.nconst == 0, "this model takes %d constants: launch it with " entry, (m)->d.nconst)

extern "C" int mc3b_user_model_chisq_ex(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                        int64_t nchains, const void* x, const void* data, const void* invsig,
                                        int64_t n, double* partial, int64_t ldpartial, int nsplit,
                                        const mc3b_chisq_opts_t* opts, void* stream) {
    MC3B_CHECK_ARG(m && x, "null pointer");
    MC3B_CHECK_ARG(m->d.ninputs == 1, "this model takes %d inputs: launch it with mc3b_user_model_chisq_inputs",
                   m->d.ninputs);
    MC3B_NO_CONSTS(m, "mc3b_user_model_chisq_consts");
    return user_chisq(m, params, ldp, nchains, &x, nullptr, data, invsig, n, partial, ldpartial, nsplit, opts, stream);
}

extern "C" int mc3b_user_model_chisq_inputs(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                            int64_t nchains, const void* const* xs, int nx, const void* data,
                                            const void* invsig, int64_t n, double* partial, int64_t ldpartial,
                                            int nsplit, const mc3b_chisq_opts_t* opts, void* stream) {
    MC3B_CHECK_ARG(m && xs, "null pointer");
    MC3B_CHECK_ARG(nx == m->d.ninputs, "this model takes %d inputs, got %d", m->d.ninputs, nx);
    MC3B_NO_CONSTS(m, "mc3b_user_model_chisq_consts");
    return user_chisq(m, params, ldp, nchains, xs, nullptr, data, invsig, n, partial, ldpartial, nsplit, opts, stream);
}

extern "C" int mc3b_user_model_chisq_consts(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                            int64_t nchains, const void* const* xs, int nx, const void* consts,
                                            int nk, const void* data, const void* invsig, int64_t n, double* partial,
                                            int64_t ldpartial, int nsplit, const mc3b_chisq_opts_t* opts,
                                            void* stream) {
    MC3B_CHECK_ARG(m && xs, "null pointer");
    MC3B_CHECK_ARG(nx == m->d.ninputs, "this model takes %d inputs, got %d", m->d.ninputs, nx);
    MC3B_CHECK_ARG(nk == m->d.nconst, "this model takes %d constants, got %d", m->d.nconst, nk);
    return user_chisq(m, params, ldp, nchains, xs, consts, data, invsig, n, partial, ldpartial, nsplit, opts, stream);
}

extern "C" int mc3b_user_model_eval(const mc3b_user_model_t* m, const double* params, int64_t ldp, int64_t nchains,
                                    const double* x, int64_t n, double* out, void* stream) {
    MC3B_CHECK_ARG(m && x, "bad arguments");
    MC3B_CHECK_ARG(m->d.ninputs == 1, "this model takes %d inputs: evaluate it with mc3b_user_model_eval_inputs",
                   m->d.ninputs);
    MC3B_NO_CONSTS(m, "mc3b_user_model_eval_consts");
    return user_eval(m, params, ldp, nchains, &x, nullptr, n, out, stream);
}

extern "C" int mc3b_user_model_eval_inputs(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                           int64_t nchains, const double* const* xs, int nx, int64_t n, double* out,
                                           void* stream) {
    MC3B_CHECK_ARG(m && xs, "bad arguments");
    MC3B_CHECK_ARG(nx == m->d.ninputs, "this model takes %d inputs, got %d", m->d.ninputs, nx);
    MC3B_NO_CONSTS(m, "mc3b_user_model_eval_consts");
    return user_eval(m, params, ldp, nchains, xs, nullptr, n, out, stream);
}

extern "C" int mc3b_user_model_eval_consts(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                           int64_t nchains, const double* const* xs, int nx, const double* consts,
                                           int nk, int64_t n, double* out, void* stream) {
    MC3B_CHECK_ARG(m && xs, "bad arguments");
    MC3B_CHECK_ARG(nx == m->d.ninputs, "this model takes %d inputs, got %d", m->d.ninputs, nx);
    MC3B_CHECK_ARG(nk == m->d.nconst, "this model takes %d constants, got %d", m->d.nconst, nk);
    return user_eval(m, params, ldp, nchains, xs, consts, n, out, stream);
}

extern "C" int mc3b_user_model_dwt_chisq(const mc3b_user_model_t* m, const double* params, int64_t ldp,
                                         int64_t nchains, int npars, const double* const* xs, int nx,
                                         const double* consts, int nk, const double* data, int64_t n,
                                         void* workspace, double* chisq, void* stream) {
    MC3B_CHECK_ARG(m && xs, "null pointer");
    MC3B_CHECK_ARG(m->d.dtype == MC3B_F64,
                   "the wavelet likelihood takes the fp64 module of a user model; this handle is fp32");
    MC3B_CHECK_ARG(nx == m->d.ninputs, "this model takes %d inputs, got %d", m->d.ninputs, nx);
    MC3B_CHECK_ARG(nk == m->d.nconst, "this model takes %d constants, got %d", m->d.nconst, nk);
    MC3B_CHECK_ARG(consts || m->d.nconst == 0, "null pointer (constants)");
    const DwtUserModel u = {(const void*)m->dwt[0], (const void*)m->dwt[1], (const void*)m->dwt[2], nx, m->d.nmodel,
                            xs, consts};
    return mc3b_dwt_chisq_user(u, params, ldp, nchains, npars, data, n, workspace, chisq, (cudaStream_t)stream);
}
