/*
 * bgw_jit.h -- run-time compilation of the general step kernel for ONE spec (bgw_specialize, include/bgw.h).
 *
 * The general kernel (bgw_dev.cuh, bgw_step_body) serves every sim the component API can describe; one CTA per env runs
 * at its own place in 9-16 k instructions and waits for instruction fetches most of the time (profiles/: no_instruction is
 * its top stall).  With the spec's scalars as compile-time constants the same source compiles to a third of that: every
 * dispatch on program / actor / observer / manager folds, loops get their trip counts, the shared-memory offsets become
 * immediates.  NVRTC (libnvrtc.so.12, opened with dlopen: no link-time dependency) compiles
 *
 *     #define BGW_JIT_PIN  s.H = ..; s.W = ..; ...         (every int scalar of DevSpec except E / env_offset / horizon)
 *     #define BGW_JIT_T    <threads per env>
 *     #include "bgw_dev.cuh"
 *     extern "C" __global__ void bgw_step_jit(...) { bgw_step_body<PROG, ATT>(...); }
 *
 * for sm_100a into a cubin, which is loaded through the driver API (libcuda.so.1, dlopen) into the primary context the
 * runtime API uses, and launched with cuLaunchKernel.  bgw_set_program compiles the same kernel with a user step program
 * in it (bgw_program.cuh).  Host code only; included by bgw.cu.
 */
#ifndef BGW_JIT_H_
#define BGW_JIT_H_

#include <cuda.h>          /* types and constants only: the driver is opened with dlopen, nothing links against libcuda */
#include <dlfcn.h>
#include <sys/stat.h>

#include <string>

namespace bgwjit {

typedef struct _nvrtcProgram *nvrtcProgram;

struct Nvrtc {
    void *lib = nullptr;
    int (*CreateProgram)(nvrtcProgram *, const char *, const char *, int, const char *const *, const char *const *) = nullptr;
    int (*CompileProgram)(nvrtcProgram, int, const char *const *) = nullptr;
    int (*GetCUBINSize)(nvrtcProgram, size_t *) = nullptr;
    int (*GetCUBIN)(nvrtcProgram, char *) = nullptr;
    int (*GetProgramLogSize)(nvrtcProgram, size_t *) = nullptr;
    int (*GetProgramLog)(nvrtcProgram, char *) = nullptr;
    int (*DestroyProgram)(nvrtcProgram *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    int (*Version)(int *, int *) = nullptr;
    int major = 0, minor = 0;
};

struct Driver {
    void *lib = nullptr;
    int (*ModuleLoadData)(CUmodule *, const void *) = nullptr;
    int (*ModuleGetFunction)(CUfunction *, CUmodule, const char *) = nullptr;
    int (*ModuleUnload)(CUmodule) = nullptr;
    int (*FuncSetAttribute)(CUfunction, int, int) = nullptr;
    int (*LaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, void *, void **, void **) = nullptr;
    int (*LaunchKernelEx)(const CUlaunchConfig *, CUfunction, void **, void **) = nullptr;
    int (*OccupancyMaxActiveBlocks)(int *, CUfunction, int, size_t) = nullptr;
    int (*GetErrorString)(int, const char **) = nullptr;
};

template <typename F>
inline bool sym(void *lib, const char *name, F &out)
{
    out = reinterpret_cast<F>(dlsym(lib, name));
    return out != nullptr;
}

/* $BGW_NVRTC if set; else the newest of the toolkit's copy and whatever "libnvrtc.so.12" resolves to (inside a PyTorch
 * process that is PyTorch's bundled copy, which may be older than the toolkit the library was built with: the 256-bit
 * store of the row gather needs PTX 8.8 = NVRTC 12.9; with an older one the kernels are compiled with -DBGW_NO_ST256). */
inline const char *load_nvrtc(Nvrtc &n)
{
    if (n.lib) return nullptr;
    const char *forced = getenv("BGW_NVRTC");            /* this one and no other */
    const char *names[] = {forced, "/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so.12", "libnvrtc.so"};
    for (const char *nm : names) {
        if (!nm || !*nm || (forced && *forced && nm != forced)) continue;
        void *lib = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
        if (!lib) continue;
        Nvrtc c;
        c.lib = lib;
        if (!sym(lib, "nvrtcCreateProgram", c.CreateProgram) || !sym(lib, "nvrtcCompileProgram", c.CompileProgram) ||
            !sym(lib, "nvrtcGetCUBINSize", c.GetCUBINSize) || !sym(lib, "nvrtcGetCUBIN", c.GetCUBIN) ||
            !sym(lib, "nvrtcGetProgramLogSize", c.GetProgramLogSize) || !sym(lib, "nvrtcGetProgramLog", c.GetProgramLog) ||
            !sym(lib, "nvrtcDestroyProgram", c.DestroyProgram) || !sym(lib, "nvrtcGetErrorString", c.GetErrorString) ||
            !sym(lib, "nvrtcVersion", c.Version) || c.Version(&c.major, &c.minor) != 0) { dlclose(lib); continue; }
        if (!n.lib || c.major * 100 + c.minor > n.major * 100 + n.minor) { if (n.lib) dlclose(n.lib); n = c; }
        else dlclose(lib);
    }
    if (!n.lib) return "no usable libnvrtc.so.12 ($BGW_NVRTC, /usr/local/cuda/lib64, the loader path)";
    if (n.major * 100 + n.minor < 1208) { dlclose(n.lib); n = Nvrtc(); return "libnvrtc is older than 12.8: it cannot compile for sm_100a"; }
    return nullptr;
}

inline const char *load_driver(Driver &d)
{
    if (d.lib) return nullptr;
    if (!(d.lib = dlopen("libcuda.so.1", RTLD_NOW | RTLD_LOCAL))) return "libcuda.so.1 not found";
    if (!sym(d.lib, "cuModuleLoadData", d.ModuleLoadData) || !sym(d.lib, "cuModuleGetFunction", d.ModuleGetFunction) ||
        !sym(d.lib, "cuModuleUnload", d.ModuleUnload) || !sym(d.lib, "cuFuncSetAttribute", d.FuncSetAttribute) ||
        !sym(d.lib, "cuLaunchKernel", d.LaunchKernel) || !sym(d.lib, "cuLaunchKernelEx", d.LaunchKernelEx) ||
        !sym(d.lib, "cuOccupancyMaxActiveBlocksPerMultiprocessor", d.OccupancyMaxActiveBlocks) || !sym(d.lib, "cuGetErrorString", d.GetErrorString)) {
        dlclose(d.lib); d.lib = nullptr;
        return "libcuda.so.1 lacks an entry point";
    }
    return nullptr;
}

inline Nvrtc &nvrtc() { static Nvrtc n; return n; }
inline Driver &driver() { static Driver d; return d; }

/* directory of the shared object this code lives in (= abmarl_b200/csrc: the kernel sources sit next to libbgw.so) */
inline std::string library_dir()
{
    Dl_info info;
    static int anchor;
    if (!dladdr((void *)&anchor, &info) || !info.dli_fname) return ".";
    std::string p(info.dli_fname);
    const size_t k = p.find_last_of('/');
    return k == std::string::npos ? std::string(".") : p.substr(0, k);
}

inline bool read_file(const std::string &path, std::string &out)
{
    FILE *fp = fopen(path.c_str(), "rb");
    if (!fp) return false;
    char buf[1 << 16];
    size_t n;
    out.clear();
    while ((n = fread(buf, 1, sizeof(buf), fp)) > 0) out.append(buf, n);
    fclose(fp);
    return true;
}

inline unsigned long long fnv1a(const std::string &s, unsigned long long h = 1469598103934665603ull)
{
    for (unsigned char c : s) { h ^= c; h *= 1099511628211ull; }
    return h;
}

/* the statements that overwrite the spec's scalars at the top of bgw_step_body */
inline std::string pin_statements(const DevSpec &d, bool has_init_ammo)
{
    std::string s;
    char b[96];
#define PIN(f) do { snprintf(b, sizeof(b), "s." #f "=%d;", (int)d.f); s += b; } while (0)
    PIN(H); PIN(W); PIN(HW); PIN(A); PIN(L);
    PIN(program); PIN(move_actor); PIN(attack_actor); PIN(observer); PIN(observe_self); PIN(done_mask); PIN(manager); PIN(ravel);
    PIN(no_overlap); PIN(stacked); PIN(auto_reset);
    PIN(max_enc); PIN(n_blk); PIN(obs_h); PIN(obs_w); PIN(obs_c); PIN(obs_stride); PIN(nchunks);
    PIN(a_nav); PIN(a_target); PIN(a_pacman); PIN(has_food);
    for (int k = 0; k < 10; ++k) { snprintf(b, sizeof(b), "s.a_script[%d]=%d;", k, d.a_script[k]); s += b; }
    PIN(hw_words); PIN(n_var); PIN(randomize_placement_order); PIN(tpl_error); PIN(slot_mask); PIN(mask_words); PIN(mask_batch);
    PIN(parallel_actors); PIN(act_words); PIN(ammo_offset); PIN(n_ammo); PIN(position_offset); PIN(obs_cells); PIN(n_dyn_blk);
    PIN(o_head); PIN(o_slot); PIN(o_cell); PIN(o_next); PIN(o_flags); PIN(o_enc); PIN(o_klass); PIN(o_tmp); PIN(o_racc); PIN(o_act);
    PIN(o_ragent); PIN(o_plist); PIN(o_pstate); PIN(o_avail); PIN(o_mask); PIN(o_ctr); PIN(o_csum); PIN(smem_bytes);
#undef PIN
    if (!d.static_mask) s += "s.static_mask=nullptr;";
    if (!has_init_ammo) s += "s.init_ammo=nullptr;";
    return s;
}

struct Kernel {
    CUmodule module = nullptr;
    CUfunction function = nullptr;
};

/* Compile `src` (or fetch its cubin from cache_dir) and load the kernel `name` with `smem` bytes of dynamic shared memory.
 * Returns nullptr on success, else a message (static or in `msg`). */
inline const char *compile_and_load(std::string src, const char *name, int smem, const char *cache_dir, Kernel &out, std::string &msg)
{
    if (const char *e = load_driver(driver())) return e;
    const std::string dir = library_dir(), inc = dir + "/../../include";
    std::string dev, fst, prg, hdr, phl, sti, pgh;
    if (!read_file(dir + "/bgw_dev.cuh", dev) || !read_file(dir + "/bgw_fast.cuh", fst) || !read_file(dir + "/bgw_program.cuh", prg) ||
        !read_file(inc + "/bgw.h", hdr) || !read_file(inc + "/bgw_philox.h", phl) || !read_file(inc + "/bgw_stdint.h", sti) ||
        !read_file(inc + "/bgw_program.h", pgh)) {
        msg = "the kernel sources (bgw_dev.cuh, bgw_fast.cuh, bgw_program.cuh, include/bgw*.h) are not next to the library in " + dir;
        return msg.c_str();
    }
    const unsigned long long key = fnv1a(pgh, fnv1a(sti, fnv1a(phl, fnv1a(hdr, fnv1a(prg, fnv1a(fst, fnv1a(dev, fnv1a(src))))))));
    std::string cubin, cache_path;
    if (cache_dir && *cache_dir) {
        char nm[64];
        snprintf(nm, sizeof(nm), "/bgw_jit_%016llx.cubin", key);
        cache_path = std::string(cache_dir) + nm;
        read_file(cache_path, cubin);
    }
    bool from_cache = !cubin.empty();
    for (int attempt = 0;; ++attempt) {
        if (cubin.empty()) {
            if (const char *e = load_nvrtc(nvrtc())) return e;
            Nvrtc &n = nvrtc();
            nvrtcProgram prog = nullptr;
            int rc = n.CreateProgram(&prog, src.c_str(), "bgw_jit.cu", 0, nullptr, nullptr);
            if (rc) { msg = std::string("nvrtcCreateProgram: ") + n.GetErrorString(rc); return msg.c_str(); }
            const std::string i1 = "-I" + dir, i2 = "-I" + inc;
            const char *opts[] = {"--gpu-architecture=sm_100a", "-std=c++17", "--fmad=false", i1.c_str(), i2.c_str(), "-I/usr/local/cuda/include", "-lineinfo",
                                  "-DBGW_NO_ST256"};   /* the last one only with an NVRTC that predates PTX 8.8 */
            const int nopt = (int)(sizeof(opts) / sizeof(opts[0])) - (n.major * 100 + n.minor >= 1209 ? 1 : 0);
            rc = n.CompileProgram(prog, nopt, opts);
            if (rc) {
                size_t ln = 0;
                n.GetProgramLogSize(prog, &ln);
                std::string log(ln, '\0');
                if (ln) n.GetProgramLog(prog, &log[0]);
                msg = std::string("nvrtcCompileProgram: ") + n.GetErrorString(rc) + "\n" + log.substr(0, 1500);
                n.DestroyProgram(&prog);
                return msg.c_str();
            }
            size_t cn = 0;
            n.GetCUBINSize(prog, &cn);
            cubin.resize(cn);
            n.GetCUBIN(prog, &cubin[0]);
            n.DestroyProgram(&prog);
            if (!cache_path.empty()) {                    /* best effort: written under a temporary name, then renamed */
                mkdir(cache_dir, 0755);
                const std::string tmp = cache_path + ".tmp";
                if (FILE *fp = fopen(tmp.c_str(), "wb")) {
                    const bool ok = fwrite(cubin.data(), 1, cubin.size(), fp) == cubin.size();
                    fclose(fp);
                    if (ok) rename(tmp.c_str(), cache_path.c_str()); else remove(tmp.c_str());
                }
            }
        }
        Driver &c = driver();
        const char *es = nullptr;
        int rc = c.ModuleLoadData(&out.module, cubin.data());
        if (!rc) {
            rc = c.ModuleGetFunction(&out.function, out.module, name);
            if (!rc) rc = c.FuncSetAttribute(out.function, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, smem);
            if (!rc) break;
            c.ModuleUnload(out.module);
        }
        out = Kernel();
        if (from_cache && attempt == 0) {                 /* a damaged or stale cache entry: compile afresh, once */
            from_cache = false;
            cubin.clear();
            remove(cache_path.c_str());
            continue;
        }
        c.GetErrorString(rc, &es);
        msg = std::string("loading ") + name + ": " + (es ? es : "?");
        return msg.c_str();
    }
    return nullptr;
}

/* the general step kernel for one spec; with `program` (a user step program, include/bgw_program.h) compiled into it */
inline const char *build(const DevSpec &d, bool has_init_ammo, int threads, const char *cache_dir, Kernel &out, std::string &msg,
                         const char *program = nullptr)
{
    char head[1024];
    snprintf(head, sizeof(head), "#define BGW_JIT_T %d\n#define BGW_JIT_PIN ", threads);
    std::string src = std::string(program ? "#define BGW_USER_PROGRAM\n" : "") + head + pin_statements(d, has_init_ammo) +
                      "\n#include \"bgw_dev.cuh\"\n";
    if (program)   /* the program's diagnostics name its own lines */
        src += std::string("#include \"bgw_program.cuh\"\n#line 1 \"program\"\n") + program +
               "\n#define BGWP_AFTER_PROGRAM\n#include \"bgw_program.cuh\"\n";
    snprintf(head, sizeof(head),
             "extern \"C\" __global__ void __launch_bounds__(%d) bgw_step_jit(const DevSpec s_in, const BgwState st, const uint32_t *actions, "
             "const int16_t *order, int8_t *obs, float *reward, uint8_t *done, uint8_t *all_done)\n"
             "{ bgw_step_body<%d, %d>(s_in, st, actions, order, obs, reward, done, all_done); }\n",
             threads, d.program, d.attack_actor);
    src += head;
    return compile_and_load(src, "bgw_step_jit", d.smem_bytes, cache_dir, out, msg);
}

/* the specialised team-battle kernel with THIS spec's shape as its compile-time shape (bgw_fast.cuh: FastStaticC5 / C2 are
 * the two shapes the library ships; every other sim runs the run-time-shape instantiation, 2.4 x the instructions) */
inline const char *build_fast(const DevSpec &q, const FastSpec &f, int threads, int lb_n, const char *cache_dir, Kernel &out, std::string &msg)
{
    char b[1536];
    snprintf(b, sizeof(b),
             "#include \"bgw_dev.cuh\"\n#include \"bgw_fast.cuh\"\n"
             "struct FastStaticJit {\n    static constexpr bool is_static = true;\n"
             "    static constexpr int A = %d, L = %d, H = %d, W = %d, P = %d, PL = %d, PW = %d, PH = %d, obs_stride = %d, nchunks = %d,\n"
             "        obs_h = %d, view = %d, move_actor = %d, ravel = %d, observe_self = %d, done_mask = %d, max_enc = %d, simd_ok = %d,\n"
             "        async_ok = %d, slots = %d, T = %d, att = %d, identity = %d, can_mix = %d, acc_lt1 = %d, rpo = %d, LB_T = %d, LB_N = %d;\n};\n"
             "extern \"C\" __global__ void __launch_bounds__(%d, %d) bgw_step_fast_jit(const DevSpec s_in, const FastSpec f_in, const BgwState st, "
             "const uint32_t *actions, uint32_t *sampled, const int16_t *order, int8_t *obs, float *reward, uint8_t *done, uint8_t *all_done)\n"
             "{ bgw_step_fast_body<FastStaticJit, %s>(s_in, f_in, st, actions, sampled, order, obs, reward, done, all_done); }\n",
             q.A, q.L, q.H, q.W, f.P, f.PL, f.PW, f.PH, q.obs_stride, q.nchunks, q.obs_h, f.uniform_view, q.move_actor, q.ravel,
             q.observe_self, q.done_mask, q.max_enc, f.simd_ok, f.async_ok, q.slot_mask + 1, threads, f.uniform_att, f.identity_learners,
             f.can_mix, f.acc_lt1, q.randomize_placement_order, threads, lb_n, threads, lb_n, f.head_elem == 1 ? "uint8_t" : "uint16_t");
    return compile_and_load(b, "bgw_step_fast_jit", f.smem_bytes, cache_dir, out, msg);
}

}   // namespace bgwjit

#endif /* BGW_JIT_H_ */
