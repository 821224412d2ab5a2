// Verifier statistics, per-candidate scores and first-index argmax
// and (segmented) top-k (search/verifier.py:45-66, 207-248, 262-287; search/search_algorithm.py:79-81); the two
// ends of the denoising verifier around its UNet pass (level inputs, per-candidate denoising error); systematic
// resampling of Feynman-Kac particles; the rank ensemble of several verifiers' scores.
// All reductions are warp-shuffle + one shared-memory hop.
#include "its_common.cuh"

namespace its {

__device__ __forceinline__ float block_sum(float v, float* s_red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  float t = (lane < nw) ? s_red[lane] : 0.f;
  t = warp_sum(t);
  return t;  // every thread of every warp holds the total
}
__device__ __forceinline__ float block_min(float v, float* s_red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  v = warp_min(v);
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  float t = (lane < nw) ? s_red[lane] : INFINITY;
  t = warp_min(t);
  return t;
}

// One CTA per image.  stats[img] = {mean, unbiased var, min, |pooled|_2 (0 without feats)};
// feats[img][C*64] = L2-normalised adaptive 8x8 average pool (may be NULL).
__global__ void __launch_bounds__(256) image_stats_kernel(float* __restrict__ stats,
                                                          float* __restrict__ feats,
                                                          const float* __restrict__ images, int C,
                                                          int H, int W) {
  pdl_prologue();
  __shared__ float s_red[32];
  __shared__ float s_feat[4 * 64];
  const int img = blockIdx.x, tid = threadIdx.x;
  const int n = C * H * W;
  const float* x = images + (long long)img * n;
  float s = 0.f, mn = INFINITY;
  for (int i = tid; i < n; i += blockDim.x) {
    const float v = x[i];
    s += v;
    mn = fminf(mn, v);
  }
  const float mean = block_sum(s, s_red) / (float)n;
  mn = block_min(mn, s_red);
  float m2 = 0.f;
  for (int i = tid; i < n; i += blockDim.x) {
    const float d = x[i] - mean;
    m2 = fmaf(d, d, m2);
  }
  m2 = block_sum(m2, s_red);
  if (tid == 0) {
    float4 o = make_float4(mean, m2 / (float)(n - 1), mn, 0.f);
    reinterpret_cast<float4*>(stats)[img] = o;
  }
  if (feats == nullptr) return;
  // adaptive_avg_pool2d -> (8, 8): window [floor(i*H/8), ceil((i+1)*H/8))
  const int nf = C * 64;
  float sq = 0.f;
  for (int f = tid; f < nf; f += blockDim.x) {
    const int c = f >> 6, i = (f >> 3) & 7, j = f & 7;
    const int y0 = (i * H) / 8, y1 = ((i + 1) * H + 7) / 8;
    const int x0 = (j * W) / 8, x1 = ((j + 1) * W + 7) / 8;
    float a = 0.f;
    for (int yy = y0; yy < y1; ++yy)
      for (int xx = x0; xx < x1; ++xx) a += x[((long long)c * H + yy) * W + xx];
    a /= (float)((y1 - y0) * (x1 - x0));
    s_feat[f] = a;
    sq = fmaf(a, a, sq);
  }
  sq = block_sum(sq, s_red);
  if (tid == 0) stats[(long long)img * 4 + 3] = sqrtf(sq);  // norm of the pooled vector
  const float inv = 1.0f / fmaxf(sqrtf(sq), 1e-12f);         // F.normalize eps
  for (int f = tid; f < nf; f += blockDim.x) feats[(long long)img * nf + f] = s_feat[f] * inv;
}

// One warp per candidate.
__global__ void __launch_bounds__(128) candidate_scores_kernel(float* __restrict__ scores,
                                                               const float* __restrict__ stats,
                                                               const float* __restrict__ feats,
                                                               int n_cand, int per_cand,
                                                               int feat_dim, int kind) {
  pdl_prologue();
  const int cand = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (cand >= n_cand) return;
  const float4* st = reinterpret_cast<const float4*>(stats) + (long long)cand * per_cand;
  float score;
  if (kind == 0) {
    float v = 0.f;
    for (int b = lane; b < per_cand; b += 32) v += st[b].y;
    v = warp_sum(v) / (float)per_cand;
    score = 1.0f / (1.0f + v);
  } else if (kind == 1) {
    float mn = INFINITY, sd = 0.f;
    for (int b = lane; b < per_cand; b += 32) {
      mn = fminf(mn, st[b].z);
      sd += sqrtf(st[b].y);
    }
    mn = warp_min(mn);
    sd = warp_sum(sd) / (float)per_cand;
    if (mn < 0.f) sd *= 0.5f;  // std((x+1)/2) = std(x)/2
    score = sd + sd;           // color_diversity + contrast are the same quantity
  } else {
    const float* f = feats + (long long)cand * per_cand * feat_dim;
    float acc = 0.f;
    const int pairs = per_cand * per_cand;
    for (int pr = 0; pr < pairs; ++pr) {
      const int i = pr / per_cand, j = pr - i * per_cand;
      if (i == j) continue;
      float d = 0.f;
      for (int e = lane; e < feat_dim; e += 32) d = fmaf(f[(long long)i * feat_dim + e], f[(long long)j * feat_dim + e], d);
      acc += warp_sum(d);
    }
    const int cnt = pairs - per_cand;
    score = (cnt > 0) ? acc / (float)cnt : __int_as_float(0x7fc00000);  // mean of empty = NaN
  }
  if (lane == 0) scores[cand] = score;
}

struct Best { float v; int i; };
__device__ __forceinline__ Best better(Best a, Best b) {
  // strict '>' with first index on ties; i < 0 means "none yet"
  if (b.i < 0) return a;
  if (a.i < 0) return b;
  if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
  return a;
}

__global__ void __launch_bounds__(1024) argmax_first_kernel(int* __restrict__ idx_out,
                                                            float* __restrict__ val_out,
                                                            const float* __restrict__ scores, int n) {
  pdl_prologue();
  __shared__ float s_v[32];
  __shared__ int s_i[32];
  Best b = {-INFINITY, -1};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = scores[i];
    if (v > b.v) { b.v = v; b.i = i; }  // NaN and -inf never win, ties keep the earlier index
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Best t = {__shfl_xor_sync(0xffffffffu, b.v, o), __shfl_xor_sync(0xffffffffu, b.i, o)};
    b = better(b, t);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { s_v[warp] = b.v; s_i[warp] = b.i; }
  __syncthreads();
  if (warp == 0) {
    Best t = {-INFINITY, -1};
    if (lane < (int)(blockDim.x >> 5)) { t.v = s_v[lane]; t.i = s_i[lane]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      Best u = {__shfl_xor_sync(0xffffffffu, t.v, o), __shfl_xor_sync(0xffffffffu, t.i, o)};
      t = better(t, u);
    }
    if (lane == 0) { *idx_out = t.i; *val_out = t.v; }
  }
}

// Top-k selection, same ordering rule applied k times: rank r is the first index of the largest score that comes
// after rank r-1 in the order (score descending, index ascending).  NaN and -inf never rank; ranks beyond the
// number of eligible scores get index -1.  One block per segment: block s ranks scores[s*seg_len, (s+1)*seg_len)
// and writes flat indices (s*seg_len + local) to idx_out[s*k + r].  Warp-shuffle + shared-memory reduction per rank.
__global__ void __launch_bounds__(1024) topk_first_kernel(int* __restrict__ idx_out, float* __restrict__ val_out,
                                                          const float* __restrict__ scores, int seg_len, int k) {
  pdl_prologue();
  __shared__ float s_v[32];
  __shared__ int s_i[32];
  __shared__ Best s_prev;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int base = blockIdx.x * seg_len, end = base + seg_len;   // n_seg * seg_len fits int32 (checked on the host)
  idx_out += (long long)blockIdx.x * k;
  val_out += (long long)blockIdx.x * k;
  Best prev = {INFINITY, -1};
  for (int r = 0; r < k; ++r) {
    Best b = {-INFINITY, -1};
    for (int i = base + threadIdx.x; i < end; i += blockDim.x) {
      const float v = scores[i];
      const bool after = r == 0 || v < prev.v || (v == prev.v && i > prev.i);
      if (after && v > b.v) { b.v = v; b.i = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      Best t = {__shfl_xor_sync(0xffffffffu, b.v, o), __shfl_xor_sync(0xffffffffu, b.i, o)};
      b = better(b, t);
    }
    if (lane == 0) { s_v[warp] = b.v; s_i[warp] = b.i; }
    __syncthreads();
    if (warp == 0) {
      Best t = {-INFINITY, -1};
      if (lane < (int)(blockDim.x >> 5)) { t.v = s_v[lane]; t.i = s_i[lane]; }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        Best u = {__shfl_xor_sync(0xffffffffu, t.v, o), __shfl_xor_sync(0xffffffffu, t.i, o)};
        t = better(t, u);
      }
      if (lane == 0) {
        idx_out[r] = t.i;
        val_out[r] = t.v;
        s_prev = t;
      }
    }
    __syncthreads();
    prev = s_prev;
    if (prev.i < 0) {            // nothing left: the remaining ranks are empty
      for (int q = r + 1 + threadIdx.x; q < k; q += blockDim.x) { idx_out[q] = -1; val_out[q] = -INFINITY; }
      break;
    }
  }
}

// Systematic resampling of a Feynman-Kac particle population, one CTA per segment (query).  Particle i of the
// segment has the log-potential l_i = lam * (reward_i - carried_i) (fp32, separately rounded) and the weight
// w_i = exp((double)l_i - m), m the largest finite l_i; a non-finite reward or l_i weighs 0.  Thread t owns the
// contiguous particles [t*per, (t+1)*per): its partial sums run in particle order, thread 0 scans the partials in
// thread order, so C_i = P_t + (w_a + ... + w_i) and every sum has one fixed order (no atomics).  Child j takes the
// smallest i with seg_len * C_i > (u + j) * C_last; a thread finds the children of its own particles by a binary
// search over j (the positions are monotone in j) and walks its particles once.  A position that rounding puts at
// or past C_last (the exact rule never does) goes to the last particle of non-zero weight.
constexpr int kResampleThreads = 256;

__device__ __forceinline__ double fk_weight(const float* __restrict__ reward, const float* __restrict__ carried,
                                            int i, float lam, double m) {
  const float r = reward[i];
  if (!isfinite(r)) return 0.0;
  const float l = __fmul_rn(lam, __fsub_rn(r, carried ? carried[i] : 0.f));
  return isfinite(l) ? exp((double)l - m) : 0.0;
}

__global__ void __launch_bounds__(kResampleThreads) resample_systematic_kernel(
    int* __restrict__ ancestor_out, float* __restrict__ carried_out, float* __restrict__ ess_out,
    const float* __restrict__ reward, const float* __restrict__ carried, float lam, int seg_len, uint64_t seed,
    long long round, uint32_t tag) {
  pdl_prologue();
  __shared__ double s_part[kResampleThreads], s_sq[kResampleThreads];
  __shared__ float s_max[32];
  __shared__ int s_last[32];
  __shared__ double s_total;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int base = blockIdx.x * seg_len;    // n_seg * seg_len fits int32 (checked on the host)
  reward += base;
  if (carried) carried += base;
  ancestor_out += base;
  carried_out += base;
  const int per = (seg_len + nt - 1) / nt;
  const int a = min(seg_len, tid * per), b = min(seg_len, a + per);

  // m: the largest finite log-potential (a max is exact in any order)
  float mx = -INFINITY;
  for (int i = a; i < b; ++i) {
    const float r = reward[i];
    if (!isfinite(r)) continue;
    const float l = __fmul_rn(lam, __fsub_rn(r, carried ? carried[i] : 0.f));
    if (isfinite(l)) mx = fmaxf(mx, l);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) s_max[warp] = mx;
  __syncthreads();
  mx = -INFINITY;
  for (int w = 0; w < nw; ++w) mx = fmaxf(mx, s_max[w]);
  if (mx == -INFINITY) {                    // no particle has a finite weight
    for (int j = tid; j < seg_len; j += nt) { ancestor_out[j] = -1; carried_out[j] = __int_as_float(0x7fc00000); }
    if (tid == 0) ess_out[blockIdx.x] = 0.f;
    return;
  }
  const double m = (double)mx;

  // per-thread sums in particle order, the last particle of non-zero weight
  double S = 0.0, sq = 0.0;
  int last = -1;
  for (int i = a; i < b; ++i) {
    const double w = fk_weight(reward, carried, i, lam, m);
    S += w;
    sq += w * w;
    if (w > 0.0) last = i;
  }
  s_part[tid] = S;
  s_sq[tid] = sq;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
  if (lane == 0) s_last[warp] = last;
  __syncthreads();
  if (tid == 0) {                           // exclusive scan of the partials in thread order
    double acc = 0.0, acc_sq = 0.0;
    for (int t = 0; t < nt; ++t) {
      const double v = s_part[t];
      s_part[t] = acc;
      acc += v;
      acc_sq += s_sq[t];
    }
    s_total = acc;
    ess_out[blockIdx.x] = (float)(acc * acc / acc_sq);
  }
  for (int w = 0; w < nw; ++w) last = max(last, s_last[w]);
  __syncthreads();
  const double P = s_part[tid], E = P + S, total = s_total;

  // one uniform per (seed, segment, round): 53 bits of Philox4x32-10
  uint32_t c[4] = {(uint32_t)blockIdx.x, (uint32_t)round, tag, (uint32_t)((unsigned long long)round >> 32)};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const double u = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) * 1.1102230246251565e-16;
  const double n = (double)seg_len;
  // position of child j, scaled by seg_len: (u + j) * C_last (no division: its slow path would spill)
  auto pos = [&](int j) { return (u + (double)j) * total; };
  auto first_at_least = [&](double C) {     // smallest j in [0, seg_len] with pos(j) >= seg_len * C
    const double x = n * C;
    int lo = 0, hi = seg_len;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (pos(mid) >= x) hi = mid; else lo = mid + 1;
    }
    return lo;
  };
  if (S > 0.0) {                            // children with P <= position < E fall on this thread's particles
    int j = first_at_least(P);
    const int j_end = first_at_least(E);
    double acc = 0.0;
    for (int i = a; i < b && j < j_end; ++i) {
      acc += fk_weight(reward, carried, i, lam, m);
      const double C = n * (P + acc);
      for (; j < j_end && pos(j) < C; ++j) { ancestor_out[j] = base + i; carried_out[j] = reward[i]; }
    }
  }
  for (int j = first_at_least(total) + tid; j < seg_len; j += nt) {
    ancestor_out[j] = base + last;
    carried_out[j] = reward[last];
  }
}

// Rank ensemble of V member verifiers, one CTA per segment (query).  Candidate i of the segment is eligible when
// none of its V scores is NaN or -inf; for an eligible i and member v, r_v(i) = #{eligible j: S_jv < S_iv} +
// (#{eligible j: S_jv == S_iv} - 1) / 2 (average ranks from 0, exact half-integers), and
// out_i = (sum_v w_v r_v(i)) / ((sum_v w_v) (|E| - 1)) in double, member order, separately rounded (no FMA), then
// fp32; 1 when |E| = 1, NaN for an ineligible i.  Thread t owns candidates t, t + nt, ...; the comparison partners
// stream through a tile of nt candidates in shared memory, so shared memory does not grow with seg_len.  Counts are
// per-thread integers: no atomics, and the output does not depend on the launch shape.
constexpr int kRankThreads = 256;
constexpr int kRankMaxMembers = 8;

__device__ __forceinline__ bool rank_eligible(float x) { return !(isnan(x) || x == -INFINITY); }

__global__ void __launch_bounds__(kRankThreads) rank_ensemble_kernel(float* __restrict__ out,
                                                                     const float* __restrict__ scores,
                                                                     const float* __restrict__ weights, int V,
                                                                     int seg_len) {
  pdl_prologue();
  __shared__ float s_tile[kRankThreads * kRankMaxMembers];
  __shared__ unsigned char s_ok[kRankThreads];
  const int tid = threadIdx.x, nt = blockDim.x;
  const long long base = (long long)blockIdx.x * seg_len;   // n_seg * seg_len fits int32 (checked on the host)
  scores += base * V;
  out += base;
  for (int i0 = 0; i0 < seg_len; i0 += nt) {
    const int i = i0 + tid;
    float mine[kRankMaxMembers];
    int less[kRankMaxMembers], eq[kRankMaxMembers];
    bool ok = i < seg_len;
#pragma unroll
    for (int v = 0; v < kRankMaxMembers; ++v) {
      mine[v] = (v < V && i < seg_len) ? scores[(long long)i * V + v] : 0.f;
      if (v < V) ok = ok && rank_eligible(mine[v]);
      less[v] = 0;
      eq[v] = 0;
    }
    int n_ok = 0;
    for (int j0 = 0; j0 < seg_len; j0 += nt) {
      const int cnt = min(nt, seg_len - j0);
      __syncthreads();                      // the previous tile has been read
      const float* src = scores + (long long)j0 * V;
      for (int e = tid; e < cnt * V; e += nt) s_tile[e] = src[e];
      __syncthreads();
      if (tid < cnt) {
        bool okj = true;
        for (int v = 0; v < V; ++v) okj = okj && rank_eligible(s_tile[tid * V + v]);
        s_ok[tid] = okj;
      }
      __syncthreads();
      if (!ok) continue;
      for (int jj = 0; jj < cnt; ++jj) {
        if (!s_ok[jj]) continue;
        ++n_ok;
#pragma unroll
        for (int v = 0; v < kRankMaxMembers; ++v) {
          if (v < V) {
            const float x = s_tile[jj * V + v];
            less[v] += x < mine[v];
            eq[v] += x == mine[v];
          }
        }
      }
    }
    if (i >= seg_len) continue;
    if (!ok) {
      out[i] = __int_as_float(0x7fc00000);
      continue;
    }
    if (n_ok == 1) {
      out[i] = 1.0f;
      continue;
    }
    double num = 0.0, wsum = 0.0;
    for (int v = 0; v < V; ++v) {
      double r = 0.0;
#pragma unroll
      for (int u = 0; u < kRankMaxMembers; ++u)       // register arrays: select member v without local memory
        if (u == v) r = (double)less[u] + 0.5 * (double)(eq[u] - 1);
      const double w = (double)__ldg(weights + v);
      num = __dadd_rn(num, __dmul_rn(w, r));
      wsum = __dadd_rn(wsum, w);
    }
    out[i] = (float)__ddiv_rn(num, __dmul_rn(wsum, (double)(n_ok - 1)));
  }
}

// Inputs of the denoising verifier: out[i*S + s] = a_s * x[i] + b_s * eps_tab[s] (image-major, level-minor), one
// float4 per thread, separately rounded mul / mul / add (torch's `a * x + b * eps` in fp32).
__global__ void __launch_bounds__(256) level_inputs_kernel(float* __restrict__ out, const float* __restrict__ x,
                                                           const float* __restrict__ eps_tab,
                                                           const float* __restrict__ coef, int n_levels,
                                                           long long quads_per, long long total) {
  pdl_prologue();
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < total;
       q += (long long)gridDim.x * blockDim.x) {
    const long long row = q / quads_per;
    const long long quad = q - row * quads_per;
    const long long img = row / n_levels;
    const int s = (int)(row - img * n_levels);
    const float a = __ldg(coef + 2 * s), b = __ldg(coef + 2 * s + 1);
    const float4 xv = __ldg(reinterpret_cast<const float4*>(x) + img * quads_per + quad);
    const float4 ev = __ldg(reinterpret_cast<const float4*>(eps_tab) + s * quads_per + quad);
    float4 o;
    o.x = __fadd_rn(__fmul_rn(a, xv.x), __fmul_rn(b, ev.x));
    o.y = __fadd_rn(__fmul_rn(a, xv.y), __fmul_rn(b, ev.y));
    o.z = __fadd_rn(__fmul_rn(a, xv.z), __fmul_rn(b, ev.z));
    o.w = __fadd_rn(__fmul_rn(a, xv.w), __fmul_rn(b, ev.w));
    reinterpret_cast<float4*>(out)[q] = o;
  }
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ double sq_err4(const float4 p, const float4 e) {
  const double d0 = __fsub_rn(p.x, e.x), d1 = __fsub_rn(p.y, e.y), d2 = __fsub_rn(p.z, e.z), d3 = __fsub_rn(p.w, e.w);
  return ((d0 * d0 + d1 * d1) + d2 * d2) + d3 * d3;
}

constexpr int kScoreThreads = 256;

// One CTA of kScoreThreads per candidate: D = sum over its rows (c*per_cand + b)*S + s of (eps_hat - eps_tab[s])^2,
// differences in fp32, squares and sums in double.  Thread j takes quads j, j + 256, ... of the candidate; the
// per-thread sums are combined by a fixed shuffle tree, so the order depends on nothing but the candidate's size.
// eps_u == NULL: score = -D_c / count; else (D_u - D_c) / count.  A NaN anywhere propagates to the score.
__global__ void __launch_bounds__(kScoreThreads) denoise_scores_kernel(
    float* __restrict__ scores, const float* __restrict__ eps_c, const float* __restrict__ eps_u,
    const float* __restrict__ eps_tab, int n_levels, long long rows_per_cand, long long quads_per) {
  pdl_prologue();
  __shared__ double s_c[kScoreThreads / 32], s_u[kScoreThreads / 32];
  const long long row0 = (long long)blockIdx.x * rows_per_cand;
  const long long n_q = rows_per_cand * quads_per;
  const float4* pc = reinterpret_cast<const float4*>(eps_c) + row0 * quads_per;
  const float4* pu = eps_u ? reinterpret_cast<const float4*>(eps_u) + row0 * quads_per : nullptr;
  const float4* pe = reinterpret_cast<const float4*>(eps_tab);
  double acc_c = 0.0, acc_u = 0.0;
  for (long long q = threadIdx.x; q < n_q; q += kScoreThreads) {
    const long long r = q / quads_per;
    const long long quad = q - r * quads_per;
    const int s = (int)((row0 + r) % n_levels);
    const float4 e = __ldg(pe + s * quads_per + quad);
    acc_c += sq_err4(__ldg(pc + q), e);
    if (pu) acc_u += sq_err4(__ldg(pu + q), e);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  acc_c = warp_sum_d(acc_c);
  acc_u = warp_sum_d(acc_u);
  if (lane == 0) { s_c[warp] = acc_c; s_u[warp] = acc_u; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double dc = 0.0, du = 0.0;
    for (int w = 0; w < kScoreThreads / 32; ++w) { dc += s_c[w]; du += s_u[w]; }
    const double count = (double)rows_per_cand * (double)(quads_per * 4);
    scores[blockIdx.x] = (float)((pu ? du - dc : -dc) / count);
  }
}

}  // namespace its

extern "C" int its_level_inputs(float* out, const float* x, const float* eps_tab, const float* coef, int32_t n_img,
                                int32_t n_levels, int64_t n_per, void* stream) {
  ITS_REQUIRE(out && x && eps_tab && coef, "its_level_inputs: null pointer");
  ITS_REQUIRE(n_img >= 1 && n_levels >= 1 && n_per >= 1 && n_per % 4 == 0,
              "its_level_inputs: n_img=%d n_levels=%d must be >= 1, n_per=%lld a positive multiple of 4", n_img,
              n_levels, (long long)n_per);
  const long long quads = n_per / 4, total = (long long)n_img * n_levels * quads;
  long long grid = (total + 255) / 256;
  if (grid > 148LL * 8) grid = 148LL * 8;  // 8 resident 256-thread CTAs per SM, grid-stride beyond
  ITS_LAUNCH(its::level_inputs_kernel, dim3((unsigned)grid), dim3(256), 0, its::as_stream(stream), out, x, eps_tab,
             coef, (int)n_levels, quads, total);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_denoise_scores(float* scores, const float* eps_c, const float* eps_u, const float* eps_tab,
                                  int32_t n_cand, int32_t per_cand, int32_t n_levels, int64_t n_per, void* stream) {
  ITS_REQUIRE(scores && eps_c && eps_tab, "its_denoise_scores: null pointer");
  ITS_REQUIRE(n_cand >= 1 && per_cand >= 1 && n_levels >= 1 && n_per >= 1 && n_per % 4 == 0,
              "its_denoise_scores: n_cand=%d per_cand=%d n_levels=%d must be >= 1, n_per=%lld a positive multiple "
              "of 4", n_cand, per_cand, n_levels, (long long)n_per);
  ITS_LAUNCH(its::denoise_scores_kernel, dim3((unsigned)n_cand), dim3(its::kScoreThreads), 0, its::as_stream(stream),
             scores, eps_c, eps_u, eps_tab, (int)n_levels, (long long)per_cand * n_levels, (long long)(n_per / 4));
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_image_stats(float* stats, float* feats, const float* images, int32_t n_img,
                               int32_t C, int32_t H, int32_t W, void* stream) {
  ITS_REQUIRE(stats && images, "its_image_stats: null pointer");
  ITS_REQUIRE(n_img > 0 && C > 0 && C <= 4 && H > 0 && W > 0 && (long long)C * H * W > 1,
              "its_image_stats: unsupported shape C=%d H=%d W=%d", C, H, W);
  ITS_LAUNCH(its::image_stats_kernel, dim3(n_img), dim3(256), 0, its::as_stream(stream), stats, feats, images, C, H, W);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_candidate_scores(float* scores, const float* stats, const float* feats,
                                    int32_t n_cand, int32_t per_cand, int32_t feat_dim,
                                    int32_t kind, void* stream) {
  ITS_REQUIRE(scores && stats, "its_candidate_scores: null pointer");
  ITS_REQUIRE(n_cand > 0 && per_cand > 0 && kind >= 0 && kind <= 2, "its_candidate_scores: bad arguments");
  ITS_REQUIRE(kind != 2 || (feats != nullptr && feat_dim > 0), "its_candidate_scores: kind 2 needs feats");
  const int blocks = (n_cand * 32 + 127) / 128;
  ITS_LAUNCH(its::candidate_scores_kernel, dim3(blocks), dim3(128), 0, its::as_stream(stream), scores, stats, feats, n_cand,
                                                                          per_cand, feat_dim, kind);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_argmax_first(int32_t* idx_out, float* val_out, const float* scores, int32_t n,
                                void* stream) {
  ITS_REQUIRE(idx_out && val_out && scores && n > 0, "its_argmax_first: bad arguments");
  ITS_LAUNCH(its::argmax_first_kernel, dim3(1), dim3(1024), 0, its::as_stream(stream), idx_out, val_out, scores, n);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_topk_first_segmented(int32_t* idx_out, float* val_out, const float* scores, int32_t n_seg,
                                        int32_t seg_len, int32_t k, void* stream) {
  ITS_REQUIRE(idx_out && val_out && scores, "its_topk_first_segmented: null pointer");
  ITS_REQUIRE(n_seg > 0 && seg_len > 0 && k > 0, "its_topk_first_segmented: n_seg=%d seg_len=%d k=%d must be >= 1",
              n_seg, seg_len, k);
  ITS_REQUIRE((long long)n_seg * seg_len <= INT32_MAX,
              "its_topk_first_segmented: n_seg * seg_len = %lld exceeds int32", (long long)n_seg * seg_len);
  // one warp per 32 scores of a segment, up to 32 warps: search populations are tens to hundreds per segment
  const int threads = seg_len >= 1024 ? 1024 : (seg_len + 31) / 32 * 32;
  ITS_LAUNCH(its::topk_first_kernel, dim3(n_seg), dim3(threads), 0, its::as_stream(stream), idx_out, val_out, scores,
             seg_len, k);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_resample_systematic(int32_t* ancestor_out, float* carried_out, float* ess_out, const float* reward,
                                       const float* carried_in, float lam, int32_t n_seg, int32_t seg_len,
                                       uint64_t seed, int64_t round, int32_t tag, void* stream) {
  ITS_REQUIRE(ancestor_out && carried_out && ess_out && reward, "its_resample_systematic: null pointer");
  ITS_REQUIRE(n_seg >= 1 && seg_len >= 1, "its_resample_systematic: n_seg=%d seg_len=%d must be >= 1", n_seg,
              seg_len);
  ITS_REQUIRE((long long)n_seg * seg_len <= INT32_MAX, "its_resample_systematic: n_seg * seg_len = %lld exceeds int32",
              (long long)n_seg * seg_len);
  ITS_REQUIRE(isfinite(lam) && lam >= 0.f, "its_resample_systematic: lam=%g must be finite and >= 0", (double)lam);
  const int threads = seg_len >= its::kResampleThreads ? its::kResampleThreads : (seg_len + 31) / 32 * 32;
  ITS_LAUNCH(its::resample_systematic_kernel, dim3(n_seg), dim3(threads), 0, its::as_stream(stream), ancestor_out,
             carried_out, ess_out, reward, carried_in, lam, (int)seg_len, seed, (long long)round, (uint32_t)tag);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_rank_ensemble(float* out, const float* scores, const float* weights, int32_t n_members,
                                 int32_t n_seg, int32_t seg_len, void* stream) {
  ITS_REQUIRE(out && scores && weights, "its_rank_ensemble: null pointer");
  ITS_REQUIRE(n_members >= 1 && n_members <= its::kRankMaxMembers, "its_rank_ensemble: n_members=%d outside [1, %d]",
              n_members, its::kRankMaxMembers);
  ITS_REQUIRE(n_seg >= 1 && seg_len >= 1, "its_rank_ensemble: n_seg=%d seg_len=%d must be >= 1", n_seg, seg_len);
  ITS_REQUIRE((long long)n_seg * seg_len <= INT32_MAX, "its_rank_ensemble: n_seg * seg_len = %lld exceeds int32",
              (long long)n_seg * seg_len);
  const int threads = seg_len >= its::kRankThreads ? its::kRankThreads : (seg_len + 31) / 32 * 32;
  ITS_LAUNCH(its::rank_ensemble_kernel, dim3(n_seg), dim3(threads), 0, its::as_stream(stream), out, scores, weights,
             (int)n_members, (int)seg_len);
  ITS_CHECK_LAUNCH();
  return ITS_OK;
}

extern "C" int its_topk_first(int32_t* idx_out, float* val_out, const float* scores, int32_t n, int32_t k,
                              void* stream) {
  ITS_REQUIRE(idx_out && val_out && scores && n > 0 && k > 0, "its_topk_first: bad arguments");
  return its_topk_first_segmented(idx_out, val_out, scores, 1, n, k, stream);
}
