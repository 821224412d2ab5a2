// Fused DDPM ancestral update: guidance mix + posterior mean + noise + NaN flag
// + final clip, one coalesced float4 pass (HBM-bound).  See include/its_b200.h.
#include "its_common.cuh"
#include <stdlib.h>
#include <stdarg.h>

namespace its {

static int g_pdl = -1;   // -1: read ITS_PDL from the environment on first use
// Programmatic dependent launch mode: 0 = off, 1 = every launch, 2 = small kernels only, 3 = tap-GEMMs
// only (default).  Measured on one UNet pass (config A, 64 images): off 1914 us, all 1990 us, small
// kernels only 2018 us, tap-GEMMs only 1853 us — a GEMM grid launched early sets up while the
// GroupNorm before it drains, whereas a GroupNorm grid launched early cannot become resident next to
// a persistent GEMM CTA and only pays the griddepcontrol latency.
bool pdl_enabled(int kind) {
  if (g_pdl < 0) {
    const char* e = getenv("ITS_PDL");
    g_pdl = (e != nullptr && e[0] >= '0' && e[0] <= '4') ? (e[0] - '0') : 3;
  }
  // 4 (experiment, round 2): tap-GEMMs and GroupNorm-apply, the latter WITHOUT an early trigger of its own
  // dependents: 1 942 us per config-A pass against 1 757 for mode 3 (the GEMM behind the GroupNorm loses its
  // early launch, and an early-launched GroupNorm grid is itself no faster) — every combination that puts the
  // attribute on the GroupNorm launches loses (re-measured this round: 3 -> 1 757, 1 -> 1 870, 0 -> 1 884, 2 -> 1 948)
  if (g_pdl == 4) return kind == 1 || kind == 2;
  return g_pdl == 1 || (g_pdl == 2 && kind != 1) || (g_pdl == 3 && kind == 1);
}

// Swish formulation of the GroupNorm(+Swish) kernels: tanh (one special-function operation per element, default)
// or exact (exp2 + reciprocal); ITS_SWISH=exact|tanh in the environment.
bool swish_tanh_enabled() {
  static int mode = -1;
  if (mode < 0) {
    const char* e = getenv("ITS_SWISH");
    mode = (e != nullptr && e[0] == 'e') ? 0 : 1;
  }
  return mode == 1;
}

char* err_buf() {
  static thread_local char buf[512] = "";
  return buf;
}
int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}

// clip to [-1, 1] that keeps NaN (torch.clip semantics), so a diverged x0 prediction never ranks
__device__ __forceinline__ float clip1_keep_nan(float v) { return v != v ? v : fminf(fmaxf(v, -1.f), 1.f); }

// One thread handles 4 consecutive elements of one image (n_per_img % 4 == 0),
// which is also one Philox counter.  Grid-stride over quads.
// kX0 = false: its_ddpm_step (the trailing three arguments are unused).  kX0 = true: its_ddpm_step_x0 — the
// candidate base is read from *cand_dev and, when x0_out != NULL, the x0 prediction of the same mixed eps,
// clip(r1[t]*x - r2[t]*eps, -1, 1) with {r1, r2} = x0_coef[t], is written to x0_out.
// kWImg = true: its_ddpm_step_x0_w — image img of the launch mixes with the pair {w, 1 + w} = w_img[img] instead of
// the scalar arguments w, opw.  w_img is the last parameter, so the other instantiations keep their parameter
// offsets and machine code.
template <bool kX0, bool kWImg = false>
__global__ void __launch_bounds__(256) ddpm_step_kernel(
    float* __restrict__ x, const float* __restrict__ eps_c, const float* __restrict__ eps_u,
    const float* __restrict__ noise, long long noise_t_stride, long long n_img, long long quads_per_img,
    const float* __restrict__ coef, const int* __restrict__ t_dev, float w, float opw, uint64_t seed,
    long long cand_id0, int* __restrict__ nan_flag, int clip_last, float* __restrict__ x0_out,
    const float* __restrict__ x0_coef, const long long* __restrict__ cand_dev, const float* __restrict__ w_img) {
  pdl_prologue();
  const int t = *t_dev;
  const float4 cf = *reinterpret_cast<const float4*>(coef + 4 * (long long)t);
  const float c1 = cf.x, c2 = cf.y, sigma = (t > 0) ? cf.z : 0.0f;
  float r1 = 0.f, r2 = 0.f;
  if constexpr (kX0) {
    cand_id0 = *cand_dev;
    if (x0_out != nullptr) {
      const float2 r = *reinterpret_cast<const float2*>(x0_coef + 2 * (long long)t);
      r1 = r.x;
      r2 = r.y;
    }
  }
  const bool last = (t == 0) && clip_last;
  const long long total = n_img * quads_per_img;
  if (noise != nullptr) noise += (long long)t * noise_t_stride;
  bool bad = false;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < total;
       q += (long long)gridDim.x * blockDim.x) {
    const long long img = q / quads_per_img;
    const uint32_t quad = (uint32_t)(q - img * quads_per_img);
    float4 xv = reinterpret_cast<const float4*>(x)[q];
    float4 e = __ldg(reinterpret_cast<const float4*>(eps_c) + q);
    if (eps_u != nullptr) {
      float4 u = __ldg(reinterpret_cast<const float4*>(eps_u) + q);
      float mw = w, mopw = opw;
      if constexpr (kWImg) {   // 8 B per image: the pairs of a launch stay in L1
        const float2 p = __ldg(reinterpret_cast<const float2*>(w_img) + img);
        mw = p.x;
        mopw = p.y;
      }
      // (1 + w) * eps - w * nonEps: separately rounded mul, mul, sub like the
      // reference's three eager ops (no FMA contraction), so injected-noise runs
      // can match it bit for bit.
      e.x = __fsub_rn(__fmul_rn(mopw, e.x), __fmul_rn(mw, u.x));
      e.y = __fsub_rn(__fmul_rn(mopw, e.y), __fmul_rn(mw, u.y));
      e.z = __fsub_rn(__fmul_rn(mopw, e.z), __fmul_rn(mw, u.z));
      e.w = __fsub_rn(__fmul_rn(mopw, e.w), __fmul_rn(mw, u.w));
    }
    if constexpr (kX0) {
      if (x0_out != nullptr) {
        float4 p;
        p.x = clip1_keep_nan(__fsub_rn(__fmul_rn(r1, xv.x), __fmul_rn(r2, e.x)));
        p.y = clip1_keep_nan(__fsub_rn(__fmul_rn(r1, xv.y), __fmul_rn(r2, e.y)));
        p.z = clip1_keep_nan(__fsub_rn(__fmul_rn(r1, xv.z), __fmul_rn(r2, e.z)));
        p.w = clip1_keep_nan(__fsub_rn(__fmul_rn(r1, xv.w), __fmul_rn(r2, e.w)));
        reinterpret_cast<float4*>(x0_out)[q] = p;
      }
    }
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    if (t > 0) {
      if (noise != nullptr) {
        float4 nz = __ldg(reinterpret_cast<const float4*>(noise) + q);
        z[0] = nz.x; z[1] = nz.y; z[2] = nz.z; z[3] = nz.w;
      } else {
        philox_normal4(seed, (uint64_t)(cand_id0 + img), (uint32_t)t, quad, z);
      }
    }
    float4 o;
    o.x = __fadd_rn(__fsub_rn(__fmul_rn(c1, xv.x), __fmul_rn(c2, e.x)), __fmul_rn(sigma, z[0]));
    o.y = __fadd_rn(__fsub_rn(__fmul_rn(c1, xv.y), __fmul_rn(c2, e.y)), __fmul_rn(sigma, z[1]));
    o.z = __fadd_rn(__fsub_rn(__fmul_rn(c1, xv.z), __fmul_rn(c2, e.z)), __fmul_rn(sigma, z[2]));
    o.w = __fadd_rn(__fsub_rn(__fmul_rn(c1, xv.w), __fmul_rn(c2, e.w)), __fmul_rn(sigma, z[3]));
    bad |= (o.x != o.x) | (o.y != o.y) | (o.z != o.z) | (o.w != o.w);
    if (last) {
      o.x = fminf(fmaxf(o.x, -1.f), 1.f);
      o.y = fminf(fmaxf(o.y, -1.f), 1.f);
      o.z = fminf(fmaxf(o.z, -1.f), 1.f);
      o.w = fminf(fmaxf(o.w, -1.f), 1.f);
    }
    reinterpret_cast<float4*>(x)[q] = o;
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(nan_flag, 1);
}

__global__ void __launch_bounds__(256) philox_normal_kernel(
    float* __restrict__ out, const float* __restrict__ base, int base_bcast, float scale,
    long long n_img, long long quads_per_img, uint64_t seed, long long cand_id0, uint32_t tag) {
  pdl_prologue();
  const long long total = n_img * quads_per_img;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < total;
       q += (long long)gridDim.x * blockDim.x) {
    const long long img = q / quads_per_img;
    const uint32_t quad = (uint32_t)(q - img * quads_per_img);
    float z[4];
    philox_normal4(seed, (uint64_t)(cand_id0 + img), tag, quad, z);
    float4 o = make_float4(scale * z[0], scale * z[1], scale * z[2], scale * z[3]);
    if (base != nullptr) {
      float4 b = __ldg(reinterpret_cast<const float4*>(base) + (base_bcast ? (long long)quad : q));
      o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
    }
    reinterpret_cast<float4*>(out)[q] = o;
  }
}

// Children of the path search: out[i] = a * x[parent[(child0 + i) / m]] + b * z[i], one float4 per thread,
// separately rounded mul / mul / add.  z is injected or Philox (seed, cand_id0 + child0 + i, tag, quad), the
// stream its_philox_normal gives unit cand_id0 + child0 + i.  An out-of-range parent index gives a NaN child.
__global__ void __launch_bounds__(256) path_expand_kernel(
    float* __restrict__ out, const float* __restrict__ x, const int* __restrict__ parent, int m, long long child0,
    long long n_child, long long n_parent, long long quads_per, float a, float b, const float* __restrict__ z,
    uint64_t seed, long long cand_id0, uint32_t tag) {
  pdl_prologue();
  const long long total = n_child * quads_per;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < total;
       q += (long long)gridDim.x * blockDim.x) {
    const long long c = q / quads_per;
    const uint32_t quad = (uint32_t)(q - c * quads_per);
    const long long p = __ldg(parent + (child0 + c) / m);
    float4 o;
    if (p < 0 || p >= n_parent) {
      o = make_float4(__int_as_float(0x7fffffff), __int_as_float(0x7fffffff), __int_as_float(0x7fffffff),
                      __int_as_float(0x7fffffff));
    } else {
      const float4 xv = __ldg(reinterpret_cast<const float4*>(x) + p * quads_per + quad);
      float zz[4];
      if (z != nullptr) {
        const float4 zv = __ldg(reinterpret_cast<const float4*>(z) + q);
        zz[0] = zv.x; zz[1] = zv.y; zz[2] = zv.z; zz[3] = zv.w;
      } else {
        philox_normal4(seed, (uint64_t)(cand_id0 + child0 + c), tag, quad, zz);
      }
      o.x = __fadd_rn(__fmul_rn(a, xv.x), __fmul_rn(b, zz[0]));
      o.y = __fadd_rn(__fmul_rn(a, xv.y), __fmul_rn(b, zz[1]));
      o.z = __fadd_rn(__fmul_rn(a, xv.z), __fmul_rn(b, zz[2]));
      o.w = __fadd_rn(__fmul_rn(a, xv.w), __fmul_rn(b, zz[3]));
    }
    reinterpret_cast<float4*>(out)[q] = o;
  }
}

__global__ void step_advance_kernel(int* t_dev, int delta) {
  pdl_prologue();
  *t_dev += delta;
}

static int grid_for(long long work_items, int block) {
  long long g = (work_items + block - 1) / block;
  const long long cap = 148LL * 8;  // 8 resident 256-thread CTAs per SM
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace its

extern "C" int its_version(void) { return 10000 * 0 + 100 * 1 + 0; }
extern "C" const char* its_last_error_string(void) { return its::err_buf(); }
extern "C" int its_abi_sizeof(int which) {
  return which == 0 ? (int)sizeof(its_conv_desc) : which == 1 ? (int)sizeof(its_src_t)
                                                              : (int)sizeof(its_phase_t);
}
extern "C" int its_set_pdl(int32_t enabled) {
  its::g_pdl = (enabled >= 0 && enabled <= 4) ? enabled : 3;
  return ITS_OK;
}

extern "C" int its_device_sm_count(int* out_host) {
  int dev = 0;
  ITS_CHECK_CUDA(cudaGetDevice(&dev));
  ITS_CHECK_CUDA(cudaDeviceGetAttribute(out_host, cudaDevAttrMultiProcessorCount, dev));
  return ITS_OK;
}

extern "C" int its_ddpm_step(float* x, const float* eps_c, const float* eps_u, const float* noise,
                             int64_t noise_t_stride, int64_t n_img, int64_t n_per_img, const float* coef,
                             const int32_t* t_dev, double w, uint64_t seed, int64_t cand_id0,
                             int32_t* nan_flag, int32_t clip_last, void* stream) {
  ITS_REQUIRE(x && eps_c && coef && t_dev && nan_flag, "its_ddpm_step: null pointer");
  ITS_REQUIRE(n_img > 0 && n_per_img > 0 && n_per_img % 4 == 0,
              "its_ddpm_step: n_per_img=%lld must be a positive multiple of 4", (long long)n_per_img);
  ITS_REQUIRE(noise_t_stride % 4 == 0, "its_ddpm_step: noise_t_stride must be a multiple of 4");
  const long long quads = n_per_img / 4;
  ITS_LAUNCH(its::ddpm_step_kernel<false>, dim3(its::grid_for(n_img * quads, 256)), dim3(256), 0, its::as_stream(stream), 
      x, eps_c, eps_u, noise, noise_t_stride, n_img, quads, coef, t_dev, (float)w, (float)(1.0 + w), seed,
      cand_id0,
      nan_flag, clip_last, (float*)nullptr, (const float*)nullptr, (const long long*)nullptr, (const float*)nullptr);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_ddpm_step_x0(float* x, float* x0_out, const float* eps_c, const float* eps_u, const float* noise,
                                int64_t noise_t_stride, int64_t n_img, int64_t n_per_img, const float* coef,
                                const float* x0_coef, const int32_t* t_dev, double w, uint64_t seed,
                                const int64_t* cand_dev, int32_t* nan_flag, int32_t clip_last, void* stream) {
  ITS_REQUIRE(x && eps_c && coef && t_dev && cand_dev && nan_flag, "its_ddpm_step_x0: null pointer");
  ITS_REQUIRE(x0_out == nullptr || x0_coef != nullptr, "its_ddpm_step_x0: null pointer (x0_coef with x0_out)");
  ITS_REQUIRE(n_img > 0 && n_per_img > 0 && n_per_img % 4 == 0,
              "its_ddpm_step_x0: n_per_img=%lld must be a positive multiple of 4", (long long)n_per_img);
  ITS_REQUIRE(noise_t_stride % 4 == 0, "its_ddpm_step_x0: noise_t_stride must be a multiple of 4");
  const long long quads = n_per_img / 4;
  ITS_LAUNCH(its::ddpm_step_kernel<true>, dim3(its::grid_for(n_img * quads, 256)), dim3(256), 0,
      its::as_stream(stream), x, eps_c, eps_u, noise, noise_t_stride, n_img, quads, coef, t_dev, (float)w,
      (float)(1.0 + w), seed, (long long)0, nan_flag, clip_last, x0_out, x0_coef, (const long long*)cand_dev,
      (const float*)nullptr);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_ddpm_step_x0_w(float* x, float* x0_out, const float* eps_c, const float* eps_u, const float* noise,
                                  int64_t noise_t_stride, int64_t n_img, int64_t n_per_img, const float* coef,
                                  const float* x0_coef, const int32_t* t_dev, const float* w_img, uint64_t seed,
                                  const int64_t* cand_dev, int32_t* nan_flag, int32_t clip_last, void* stream) {
  ITS_REQUIRE(x && eps_c && eps_u && coef && t_dev && w_img && cand_dev && nan_flag,
              "its_ddpm_step_x0_w: null pointer (eps_u and w_img are required)");
  ITS_REQUIRE(x0_out == nullptr || x0_coef != nullptr, "its_ddpm_step_x0_w: null pointer (x0_coef with x0_out)");
  ITS_REQUIRE(((uintptr_t)w_img & 7) == 0, "its_ddpm_step_x0_w: w_img must be 8-byte aligned ({w, 1 + w} pairs)");
  ITS_REQUIRE(n_img > 0 && n_per_img > 0 && n_per_img % 4 == 0,
              "its_ddpm_step_x0_w: n_per_img=%lld must be a positive multiple of 4", (long long)n_per_img);
  ITS_REQUIRE(noise_t_stride % 4 == 0, "its_ddpm_step_x0_w: noise_t_stride must be a multiple of 4");
  const long long quads = n_per_img / 4;
  ITS_LAUNCH((its::ddpm_step_kernel<true, true>), dim3(its::grid_for(n_img * quads, 256)), dim3(256), 0,
      its::as_stream(stream), x, eps_c, eps_u, noise, noise_t_stride, n_img, quads, coef, t_dev, 0.0f, 0.0f, seed,
      (long long)0, nan_flag, clip_last, x0_out, x0_coef, (const long long*)cand_dev, w_img);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_path_expand(float* out, const float* x, const int32_t* parent, int32_t n_sel, int32_t m,
                               int64_t child0, int64_t n_child, int64_t n_parent, int64_t n_per, float a, float b,
                               const float* z, uint64_t seed, int64_t cand_id0, int32_t tag, void* stream) {
  ITS_REQUIRE(out && x && parent, "its_path_expand: null pointer");
  ITS_REQUIRE(n_child > 0 && n_parent > 0 && n_per > 0 && n_per % 4 == 0,
              "its_path_expand: n_child=%lld n_parent=%lld must be positive, n_per=%lld a positive multiple of 4",
              (long long)n_child, (long long)n_parent, (long long)n_per);
  ITS_REQUIRE(m >= 1 && n_sel >= 1 && child0 >= 0 && child0 + n_child <= (int64_t)n_sel * m,
              "its_path_expand: children [%lld, %lld) exceed %d parents x %d children",
              (long long)child0, (long long)(child0 + n_child), n_sel, m);
  const long long quads = n_per / 4;
  ITS_LAUNCH(its::path_expand_kernel, dim3(its::grid_for(n_child * quads, 256)), dim3(256), 0,
      its::as_stream(stream), out, x, (const int*)parent, (int)m, (long long)child0, (long long)n_child,
      (long long)n_parent, quads, a, b, z, seed, (long long)cand_id0, (uint32_t)tag);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_philox_normal(float* out, const float* base, int32_t base_bcast, float scale,
                                 int64_t n_img, int64_t n_per_img, uint64_t seed, int64_t cand_id0,
                                 int32_t tag, void* stream) {
  ITS_REQUIRE(out, "its_philox_normal: null pointer");
  ITS_REQUIRE(n_img > 0 && n_per_img > 0 && n_per_img % 4 == 0,
              "its_philox_normal: n_per_img=%lld must be a positive multiple of 4", (long long)n_per_img);
  const long long quads = n_per_img / 4;
  ITS_LAUNCH(its::philox_normal_kernel, dim3(its::grid_for(n_img * quads, 256)), dim3(256), 0, its::as_stream(stream), 
      out, base, base_bcast, scale, n_img, quads, seed, cand_id0, (uint32_t)tag);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_step_advance(int32_t* t_dev, int32_t delta, void* stream) {
  ITS_REQUIRE(t_dev, "its_step_advance: null pointer");
  ITS_LAUNCH(its::step_advance_kernel, dim3(1), dim3(1), 0, its::as_stream(stream), t_dev, delta);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}
