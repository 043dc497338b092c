// jit.cpp -- see jit.h.
#include "jit.h"

#include <cuda.h>
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <mutex>
#include <vector>

#include "../../include/mecano_b200.h"
#include "rnea.cuh" // MB_PF_STAGES

namespace mb
{
namespace
{
// ---- the algorithm headers, embedded at build time (Makefile: build/embedded_headers.inc)
struct EmbeddedHeader
{
   const char *name, *text;
};
#include "build/embedded_headers.inc"

// ---- NVRTC, loaded on first use
typedef struct _nvrtcProgram *nvrtcProgram;
struct Nvrtc
{
   void *lib = nullptr;
   int (*CreateProgram)(nvrtcProgram *, const char *, const char *, int, const char *const *, const char *const *) = nullptr;
   int (*CompileProgram)(nvrtcProgram, int, const char *const *) = nullptr;
   int (*GetCUBINSize)(nvrtcProgram, size_t *) = nullptr;
   int (*GetCUBIN)(nvrtcProgram, char *) = nullptr;
   int (*GetProgramLogSize)(nvrtcProgram, size_t *) = nullptr;
   int (*GetProgramLog)(nvrtcProgram, char *) = nullptr;
   int (*DestroyProgram)(nvrtcProgram *) = nullptr;
   int (*Version)(int *, int *) = nullptr;
   const char *(*GetErrorString)(int) = nullptr;
   std::string error;
};

Nvrtc &nvrtc()
{
   static Nvrtc n;
   static std::once_flag once;
   std::call_once(once, [] {
      const char *names[] = {"libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so"};
      for (const char *nm : names)
         if ((n.lib = dlopen(nm, RTLD_NOW | RTLD_LOCAL)))
            break;
      if (!n.lib)
      {
         n.error = "libnvrtc not found (tree-specialised kernels need the CUDA toolkit's NVRTC)";
         return;
      }
#define MB_SYM(field, sym)                                    \
   *(void **)(&n.field) = dlsym(n.lib, sym);                  \
   if (!n.field) n.error = std::string("missing symbol ") + sym;
      MB_SYM(CreateProgram, "nvrtcCreateProgram")
      MB_SYM(CompileProgram, "nvrtcCompileProgram")
      MB_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
      MB_SYM(GetCUBIN, "nvrtcGetCUBIN")
      MB_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
      MB_SYM(GetProgramLog, "nvrtcGetProgramLog")
      MB_SYM(DestroyProgram, "nvrtcDestroyProgram")
      MB_SYM(Version, "nvrtcVersion")
      MB_SYM(GetErrorString, "nvrtcGetErrorString")
#undef MB_SYM
   });
   return n;
}

// ---- driver entry points through the runtime (no link-time dependency on libcuda)
struct Driver
{
   CUresult (*ModuleLoadData)(CUmodule *, const void *) = nullptr;
   CUresult (*ModuleUnload)(CUmodule) = nullptr;
   CUresult (*ModuleGetFunction)(CUfunction *, CUmodule, const char *) = nullptr;
   CUresult (*FuncGetAttribute)(int *, CUfunction_attribute, CUfunction) = nullptr;
   CUresult (*FuncSetAttribute)(CUfunction, CUfunction_attribute, int) = nullptr;
   CUresult (*LaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream, void **, void **) = nullptr;
   CUresult (*OccupancyMaxActiveBlocksPerMultiprocessor)(int *, CUfunction, int, size_t) = nullptr;
   CUresult (*GetErrorString)(CUresult, const char **) = nullptr;
   std::string error;
};

Driver &driver()
{
   static Driver d;
   static std::once_flag once;
   std::call_once(once, [] {
      auto get = [&](const char *sym, void **fn) {
         cudaDriverEntryPointQueryResult q;
         cudaError_t e = cudaGetDriverEntryPoint(sym, fn, cudaEnableDefault, &q);
         if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !*fn)
            d.error = std::string("driver entry point not available: ") + sym;
      };
      get("cuModuleLoadData", (void **)&d.ModuleLoadData);
      get("cuModuleUnload", (void **)&d.ModuleUnload);
      get("cuModuleGetFunction", (void **)&d.ModuleGetFunction);
      get("cuFuncGetAttribute", (void **)&d.FuncGetAttribute);
      get("cuFuncSetAttribute", (void **)&d.FuncSetAttribute);
      get("cuLaunchKernel", (void **)&d.LaunchKernel);
      get("cuOccupancyMaxActiveBlocksPerMultiprocessor", (void **)&d.OccupancyMaxActiveBlocksPerMultiprocessor);
      get("cuGetErrorString", (void **)&d.GetErrorString);
   });
   return d;
}

std::string cu_err(CUresult r)
{
   const char *s = nullptr;
   if (driver().GetErrorString) driver().GetErrorString(r, &s);
   return s ? s : "unknown driver error";
}

// ---- disk cache: <dir>/<hash>.cubin, hash over source + headers + NVRTC version
uint64_t fnv1a(uint64_t h, const void *p, size_t n)
{
   const unsigned char *c = (const unsigned char *)p;
   for (size_t i = 0; i < n; i++)
   {
      h ^= c[i];
      h *= 1099511628211ull;
   }
   return h;
}

// The cache holds executable code, so it is only used when nobody else can have written it: a directory owned by the
// calling user that neither group nor others may write.  Directories this function creates are private (0700).  Without
// $MECANO_B200_CACHE and without $HOME there is no trustworthy place (a shared /tmp can be pre-created by anyone): no cache.
std::string cache_dir()
{
   const char *e = getenv("MECANO_B200_CACHE");
   if (e && !*e) return ""; // empty = disabled
   std::string d;
   if (e) d = e;
   else
   {
      const char *home = getenv("HOME");
      if (!home || !*home) return "";
      d = std::string(home) + "/.cache/mecano_b200";
   }
   // mkdir -p
   for (size_t i = 1; i <= d.size(); i++)
      if (i == d.size() || d[i] == '/')
         mkdir(d.substr(0, i).c_str(), 0700);
   struct stat st;
   if (lstat(d.c_str(), &st) != 0 || !S_ISDIR(st.st_mode) || st.st_uid != geteuid() || (st.st_mode & (S_IWGRP | S_IWOTH)))
      return "";
   return d;
}

// cache entry = 32-byte header (magic, payload size, two independent 64-bit digests of the payload) + cubin: a truncated,
// corrupted or foreign file is recognised before it is handed to the driver
struct CacheHeader
{
   uint64_t magic, size, h1, h2;
};
constexpr uint64_t kCacheMagic = 0x3130424e4243424dull; // "MBCBNB01"
constexpr uint64_t kSeed1 = 1469598103934665603ull, kSeed2 = 0x9e3779b97f4a7c15ull;

bool read_file(const std::string &path, std::vector<char> &out)
{
   struct stat st;
   if (lstat(path.c_str(), &st) != 0 || !S_ISREG(st.st_mode) || st.st_uid != geteuid()) return false;
   std::ifstream f(path, std::ios::binary);
   if (!f) return false;
   std::vector<char> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
   CacheHeader hd;
   if (raw.size() <= sizeof hd) return false;
   std::memcpy(&hd, raw.data(), sizeof hd);
   const char *payload = raw.data() + sizeof hd;
   const size_t n = raw.size() - sizeof hd;
   if (hd.magic != kCacheMagic || hd.size != n || hd.h1 != fnv1a(kSeed1, payload, n) || hd.h2 != fnv1a(kSeed2, payload, n)) return false;
   out.assign(payload, payload + n);
   return true;
}

void write_file_atomic(const std::string &path, const std::vector<char> &data)
{
   const std::string tmp = path + ".tmp" + std::to_string((long)getpid());
   {
      std::ofstream f(tmp, std::ios::binary);
      if (!f) return;
      const CacheHeader hd = {kCacheMagic, (uint64_t)data.size(), fnv1a(kSeed1, data.data(), data.size()), fnv1a(kSeed2, data.data(), data.size())};
      f.write((const char *)&hd, sizeof hd);
      f.write(data.data(), (std::streamsize)data.size());
   }
   chmod(tmp.c_str(), 0600);
   rename(tmp.c_str(), path.c_str());
}

int compile(const std::string &src, std::vector<char> &cubin, std::string &err)
{
   Nvrtc &n = nvrtc();
   if (!n.error.empty())
   {
      err = n.error;
      return MECANO_B200_ERR_JIT;
   }
   std::vector<const char *> names, texts;
   for (const EmbeddedHeader &h : kEmbeddedHeaders)
   {
      names.push_back(h.name);
      texts.push_back(h.text);
   }
   nvrtcProgram prog = nullptr;
   int rc = n.CreateProgram(&prog, src.c_str(), "mb_spec.cu", (int)names.size(), texts.data(), names.data());
   if (rc != 0)
   {
      err = std::string("nvrtcCreateProgram: ") + n.GetErrorString(rc);
      return MECANO_B200_ERR_JIT;
   }
   const char *opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo"};
   rc = n.CompileProgram(prog, 3, opts);
   if (rc != 0)
   {
      size_t ls = 0;
      n.GetProgramLogSize(prog, &ls);
      std::string log(ls, '\0');
      if (ls) n.GetProgramLog(prog, &log[0]);
      err = std::string("nvrtcCompileProgram: ") + n.GetErrorString(rc) + "\n" + log.substr(0, 4000);
      n.DestroyProgram(&prog);
      return MECANO_B200_ERR_JIT;
   }
   size_t sz = 0;
   n.GetCUBINSize(prog, &sz);
   cubin.resize(sz);
   rc = n.GetCUBIN(prog, cubin.data());
   n.DestroyProgram(&prog);
   if (rc != 0 || sz == 0)
   {
      err = "nvrtcGetCUBIN failed";
      return MECANO_B200_ERR_JIT;
   }
   return MECANO_B200_OK;
}
} // namespace

int spec_compile_only(const std::string &src, size_t *cubin_bytes, std::string &err)
{
   std::vector<char> cubin;
   int rc = compile(src, cubin, err);
   if (cubin_bytes) *cubin_bytes = cubin.size();
   return rc;
}

size_t spec_smem_bytes(int algo, const MbProgram &P, int block, int tm)
{
   const int smem_slots = mb_smem_stack_slots(algo, P, tm);
   size_t bytes = sizeof(double) * ((2 * (size_t)smem_slots + mb_algo(algo).ring_rows * MB_PF_STAGES) * block);
   // a block with a TMEM stack allocates all 512 columns: keep it alone on its SM (a second block would spin in tcgen05.alloc)
   if (tm > 0)
      bytes = std::max<size_t>(bytes, 120 * 1024);
   return bytes;
}

int spec_build(int algo, const FlatTree &tree, const SpecOptions &opt, SpecKernel &out, std::string &err)
{
   Driver &d = driver();
   if (!d.error.empty())
   {
      err = d.error;
      return MECANO_B200_ERR_JIT;
   }
   const auto t0 = std::chrono::steady_clock::now();
   const std::string src = generate_source(algo, tree, opt);
   // cache key
   uint64_t h = fnv1a(1469598103934665603ull, src.data(), src.size());
   for (const EmbeddedHeader &eh : kEmbeddedHeaders)
      h = fnv1a(h, eh.text, strlen(eh.text));
   int vmaj = 0, vmin = 0;
   if (nvrtc().error.empty()) nvrtc().Version(&vmaj, &vmin);
   h = fnv1a(h, &vmaj, sizeof vmaj);
   h = fnv1a(h, &vmin, sizeof vmin);
   // second, independently seeded pass over the same bytes: a 128-bit key
   uint64_t h2 = fnv1a(kSeed2, src.data(), src.size());
   for (const EmbeddedHeader &eh : kEmbeddedHeaders)
      h2 = fnv1a(h2, eh.text, strlen(eh.text));
   h2 = fnv1a(h2, &vmaj, sizeof vmaj);
   h2 = fnv1a(h2, &vmin, sizeof vmin);
   char hex[40];
   std::snprintf(hex, sizeof hex, "%016llx%016llx", (unsigned long long)h, (unsigned long long)h2);
   const std::string dir = cache_dir();
   const std::string path = dir.empty() ? "" : dir + "/" + hex + ".cubin";
   std::vector<char> cubin;
   out.from_cache = !path.empty() && read_file(path, cubin);
   if (!out.from_cache)
   {
      int rc = compile(src, cubin, err);
      if (rc != MECANO_B200_OK) return rc;
      if (!path.empty()) write_file_atomic(path, cubin);
   }
   CUmodule mod = nullptr;
   CUresult r = d.ModuleLoadData(&mod, cubin.data());
   if (r != CUDA_SUCCESS && out.from_cache)
   {
      // stale or truncated cache entry: recompile once
      out.from_cache = false;
      int rc = compile(src, cubin, err);
      if (rc != MECANO_B200_OK) return rc;
      if (!path.empty()) write_file_atomic(path, cubin);
      r = d.ModuleLoadData(&mod, cubin.data());
   }
   if (r != CUDA_SUCCESS)
   {
      err = "cuModuleLoadData: " + cu_err(r);
      return MECANO_B200_ERR_JIT;
   }
   CUfunction fn = nullptr;
   r = d.ModuleGetFunction(&fn, mod, "mb_spec_kernel");
   if (r != CUDA_SUCCESS)
   {
      d.ModuleUnload(mod);
      err = "cuModuleGetFunction: " + cu_err(r);
      return MECANO_B200_ERR_JIT;
   }
   out.module = mod;
   out.function = fn;
   out.opt = opt;
   d.FuncGetAttribute(&out.regs, CU_FUNC_ATTRIBUTE_NUM_REGS, fn);
   d.FuncGetAttribute(&out.local_bytes, CU_FUNC_ATTRIBUTE_LOCAL_SIZE_BYTES, fn);
   d.FuncGetAttribute(&out.static_smem, CU_FUNC_ATTRIBUTE_SHARED_SIZE_BYTES, fn);
   out.smem = spec_smem_bytes(algo, tree.prog[algo], opt.block, opt.tm);
   int dev = 0, max_optin = 0, sms = 0;
   cudaGetDevice(&dev);
   cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
   cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
   if (out.smem + (size_t)out.static_smem > (size_t)max_optin)
   {
      spec_unload(out);
      err = "specialised kernel: the per-state stack does not fit in shared memory at this block size";
      return MECANO_B200_ERR_TOO_LARGE;
   }
   r = d.FuncSetAttribute(fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, max_optin - out.static_smem);
   if (r == CUDA_SUCCESS)
      r = d.OccupancyMaxActiveBlocksPerMultiprocessor(&out.blocks_per_sm, fn, opt.block, out.smem);
   if (r != CUDA_SUCCESS || out.blocks_per_sm < 1)
   {
      spec_unload(out);
      err = "specialised kernel cannot be resident (" + (r != CUDA_SUCCESS ? cu_err(r) : std::string("occupancy 0")) + ")";
      return MECANO_B200_ERR_JIT;
   }
   if (opt.tm > 0) out.blocks_per_sm = 1;
   out.grid = sms * out.blocks_per_sm;
   out.compile_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
   return MECANO_B200_OK;
}

cudaError_t spec_launch(const SpecKernel &k, const KernelArgs &a, unsigned grid, cudaStream_t stream)
{
   KernelArgs args = a;
   void *params[] = {&args};
   CUresult r = driver().LaunchKernel((CUfunction)k.function, grid, 1, 1, (unsigned)k.opt.block, 1, 1, (unsigned)k.smem, (CUstream)stream, params, nullptr);
   if (r != CUDA_SUCCESS)
      return cudaErrorLaunchFailure;
   return cudaSuccess;
}

void spec_unload(SpecKernel &k)
{
   if (k.module && driver().ModuleUnload)
      driver().ModuleUnload((CUmodule)k.module);
   k.module = nullptr;
   k.function = nullptr;
}
} // namespace mb
