// Weakly-supervised loss stack for 4-class 2D segmentation, fp32 NCHW probabilities/logits.
// Each kernel cites the reference lines (relative to /root/reference/code) whose result it reproduces.
#include "common.cuh"

namespace {

constexpr int C4 = 4;
constexpr int TPB = 256;

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// ------------------------------------------------------------------------------------------------
// K7: softmax + partial cross-entropy.  torch.softmax(outputs,1) (train_weakly_supervised_pCE_2D.py:98)
// and CrossEntropyLoss(ignore_index=4) (:81,:100) in one pass: 17 B/pixel algorithmic (4 logits, 1 label
// byte ... plus 16 B/pixel of probabilities when they are requested by a downstream regulariser).
// Each thread owns 4 consecutive pixels (float4 per class plane).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) softmax_pce_fwd_kernel(
    const float* __restrict__ logits, const uint8_t* __restrict__ label, float* __restrict__ probs,
    int HW, long long nquads, int ignore_index, float* partials, unsigned* ticket, float* out) {
  float acc[2] = {0.f, 0.f};  // nll sum, labelled count
  const int qpi = HW >> 2;
  for (long long q = blockIdx.x * (long long)TPB + threadIdx.x; q < nquads; q += (long long)gridDim.x * TPB) {
    const long long n = q / qpi;
    const int r = (int)(q - n * qpi);
    const float* base = logits + n * C4 * (long long)HW + r * 4;
    float x[C4][4];
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      float4 v = ld4(base + (long long)c * HW);
      x[c][0] = v.x; x[c][1] = v.y; x[c][2] = v.z; x[c][3] = v.w;
    }
    int lab[4] = {ignore_index, ignore_index, ignore_index, ignore_index};
    if (label != nullptr) {
      uchar4 l4 = *reinterpret_cast<const uchar4*>(label + n * (long long)HW + r * 4);
      lab[0] = l4.x; lab[1] = l4.y; lab[2] = l4.z; lab[3] = l4.w;
    }
    float p[C4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float m = fmaxf(fmaxf(x[0][j], x[1][j]), fmaxf(x[2][j], x[3][j]));
      float e[C4], s = 0.f;
#pragma unroll
      for (int c = 0; c < C4; ++c) { e[c] = expf(x[c][j] - m); s += e[c]; }
      const float inv = 1.0f / s;
#pragma unroll
      for (int c = 0; c < C4; ++c) p[c][j] = e[c] * inv;
      if (lab[j] != ignore_index && lab[j] < C4) {
        float xl = lab[j] == 0 ? x[0][j] : lab[j] == 1 ? x[1][j] : lab[j] == 2 ? x[2][j] : x[3][j];
        acc[0] += logf(s) - (xl - m);
        acc[1] += 1.f;
      }
    }
    if (probs != nullptr) {
      float* pb = probs + n * C4 * (long long)HW + r * 4;
#pragma unroll
      for (int c = 0; c < C4; ++c) st4(pb + (long long)c * HW, make_float4(p[c][0], p[c][1], p[c][2], p[c][3]));
    }
  }
  __shared__ double res[2];
  if (block_reduce_final<2, TPB>(acc, partials, ticket, res)) {
    if (threadIdx.x == 0) {
      out[0] = (float)(res[0] / res[1]);  // 0 labelled pixels -> NaN, as torch
      out[1] = (float)res[1];
    }
  }
}

// Backward of (w_ce * pCE + <gprobs, softmax>) w.r.t. logits:
//   dlogit_c = w_ce * go * (p_c - [c==label]) / count   (labelled pixels only)
//            + gs * p_c * (g_c - sum_k g_k p_k)         (softmax Jacobian applied to gprobs)
// `go` (upstream grad of the pCE scalar) is read from device memory when go_ptr != nullptr; gprobs already
// carries its own upstream scaling.
__global__ void __launch_bounds__(TPB) head_bwd_kernel(
    const float* __restrict__ probs, const uint8_t* __restrict__ label, const float* __restrict__ ce_stats,
    const float* __restrict__ go_ptr, float w_ce, const float* __restrict__ gprobs, float gs,
    int HW, long long nquads, int ignore_index, float* __restrict__ dlogits, __nv_bfloat16* __restrict__ dl_nhwc16, int dt16) {
  const int qpi = HW >> 2;
  const float go = go_ptr ? *go_ptr : 1.0f;
  const float cew = (label != nullptr && w_ce != 0.f) ? w_ce * go / ce_stats[1] : 0.f;
  const float gsc = gs;
  for (long long q = blockIdx.x * (long long)TPB + threadIdx.x; q < nquads; q += (long long)gridDim.x * TPB) {
    const long long n = q / qpi;
    const int r = (int)(q - n * qpi);
    const long long off = n * C4 * (long long)HW + r * 4;
    float p[C4][4], g[C4][4];
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      float4 v = ld4(probs + off + (long long)c * HW);
      p[c][0] = v.x; p[c][1] = v.y; p[c][2] = v.z; p[c][3] = v.w;
      if (gprobs) {
        float4 w = ld4(gprobs + off + (long long)c * HW);
        g[c][0] = w.x; g[c][1] = w.y; g[c][2] = w.z; g[c][3] = w.w;
      } else {
        g[c][0] = g[c][1] = g[c][2] = g[c][3] = 0.f;
      }
    }
    int lab[4] = {ignore_index, ignore_index, ignore_index, ignore_index};
    if (cew != 0.f) {
      uchar4 l4 = *reinterpret_cast<const uchar4*>(label + n * (long long)HW + r * 4);
      lab[0] = l4.x; lab[1] = l4.y; lab[2] = l4.z; lab[3] = l4.w;
    }
    float d[C4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float dot = 0.f;
#pragma unroll
      for (int c = 0; c < C4; ++c) dot += g[c][j] * p[c][j];
      const bool on = (lab[j] != ignore_index) && (lab[j] < C4);
#pragma unroll
      for (int c = 0; c < C4; ++c) {
        float v = gsc * p[c][j] * (g[c][j] - dot);
        if (on) v += cew * (p[c][j] - (lab[j] == c ? 1.f : 0.f));
        d[c][j] = v;
      }
    }
    if (dlogits != nullptr) {
#pragma unroll
      for (int c = 0; c < C4; ++c) st4(dlogits + off + (long long)c * HW, make_float4(d[c][0], d[c][1], d[c][2], d[c][3]));
    }
    if (dl_nhwc16 != nullptr) {
      // the executor's layout for the out_conv gradient: channels-last bf16, 4 real + 12 zero channels per pixel
      uint4* o = reinterpret_cast<uint4*>(dl_nhwc16 + (n * (long long)HW + r * 4) * 16);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 v;
        v.x = dt16 == 2 ? pack_f16(d[0][j], d[1][j]) : pack_bf16(d[0][j], d[1][j]);
        v.y = dt16 == 2 ? pack_f16(d[2][j], d[3][j]) : pack_bf16(d[2][j], d[3][j]);
        v.z = 0u; v.w = 0u;
        o[2 * j] = v;
        o[2 * j + 1] = make_uint4(0u, 0u, 0u, 0u);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K8: Gated CRF (utils/gate_crf_loss.py:20-117 for kernels_desc=[{weight,xy,rgb}], no masks, Potts).
//   k_ij = w * exp(-0.5*(|dxy|^2/sxy^2 + (I_i-I_j)^2/srgb^2)),  j in the (2R+1)^2 window, j != i
//   s_i  = sum_j k_ij y_j                (in-bounds j only: unfold zero-pads y, :89,:188)
//   loss = (sum_ij k_ij - sum_i <s_i, y_i>) / (N*H*W)                              (:63,:97-99,:116)
//   dL/dy_i = -2 s_i / (N*H*W)           (k symmetric; OOB terms carry no gradient)
// Out-of-bounds neighbours: features are zero padded (:188), so k_i,oob = w*exp(-0.5*(x_i^2+y_i^2)/sxy^2
// - 0.5*I_i^2/srgb^2) independent of the offset; it is added analytically (count * value) to sum k (F10).
// Nothing is materialised: 20 B/pixel read (y, I) + 16 B/pixel written (grad) = 36 B/pixel.
// Thread layout: lane = column, each thread owns RT vertically adjacent pixels; a neighbour value read
// from shared memory is reused for up to 2R+1 of the thread's pixels.
// ------------------------------------------------------------------------------------------------
template <int R, int RT, int WARPS>
__global__ void __launch_bounds__(32 * WARPS) gatedcrf_kernel(
    const float* __restrict__ probs, const float* __restrict__ image, float* __restrict__ gprobs,
    int N, int H, int W, float inv2sxy2 /*0.5/sxy^2*/, float inv2srgb2, float weight, float gscale /* -2*w/denom */,
    int tiles_x, int tiles_y, float* partials, unsigned* ticket, float* out, float inv_denom) {
  constexpr int D = 2 * R + 1;
  constexpr int TW = 32, TH = RT * WARPS;
  constexpr int HW_ = TW + 2 * R, HH_ = TH + 2 * R;
  constexpr float LOG2E = 1.4426950408889634f;
  extern __shared__ float smem[];
  float* sI = smem;                       // [HH_][HW_]
  float4* sY = reinterpret_cast<float4*>(smem + ((HH_ * HW_ + 3) & ~3));  // [HH_][HW_]
  __shared__ float s_lw[D * D];           // log2 of spatial weight (incl. kernel weight) per offset
  for (int i = threadIdx.x; i < D * D; i += blockDim.x) {
    int dy = i / D - R, dx = i % D - R;
    s_lw[i] = (dy == 0 && dx == 0) ? -INFINITY : (-(float)(dx * dx + dy * dy) * inv2sxy2) * LOG2E + log2f(weight);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float cI = -inv2srgb2 * LOG2E;
  float acc[2] = {0.f, 0.f};  // sum k, sum <s,y>
  const long long HW = (long long)H * W;
  const int ntiles = N * tiles_x * tiles_y;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int n = tile / (tiles_x * tiles_y);
    const int tr = tile - n * tiles_x * tiles_y;
    const int y0 = (tr / tiles_x) * TH, x0 = (tr % tiles_x) * TW;
    __syncthreads();
    for (int i = threadIdx.x; i < HH_ * HW_; i += blockDim.x) {
      const int hy = i / HW_, hx = i - hy * HW_;
      const int gy = y0 + hy - R, gx = x0 + hx - R;
      float iv = INFINITY;                 // (I_i - inf)^2 * c = -inf -> exp2 = 0 : OOB excluded from the loop
      float4 yv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
        const long long o = (long long)gy * W + gx;
        iv = image[n * HW + o];
        const float* pp = probs + n * C4 * HW + o;
        yv = make_float4(pp[0], pp[HW], pp[2 * HW], pp[3 * HW]);
      }
      sI[i] = iv;
      sY[i] = yv;
    }
    __syncthreads();
    const int ly0 = warp * RT;            // first owned row (tile-local)
    float Ic[RT];
    float4 s[RT];
    float ks[RT];
#pragma unroll
    for (int i = 0; i < RT; ++i) {
      Ic[i] = sI[(ly0 + i + R) * HW_ + lane + R];
      Ic[i] = isinf(Ic[i]) ? 0.f : Ic[i];  // own pixel OOB (ragged tile): results discarded below
      s[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      ks[i] = 0.f;
    }
#pragma unroll 1
    for (int dxi = 0; dxi < D; ++dxi) {
#pragma unroll
      for (int jr = 0; jr < RT + 2 * R; ++jr) {
        const int idx = (ly0 + jr) * HW_ + lane + dxi;
        const float Ij = sI[idx];
        const float4 yj = sY[idx];
#pragma unroll
        for (int i = 0; i < RT; ++i) {
          const int dyi = jr - i;            // = dy + R, compile-time after unrolling
          if (dyi >= 0 && dyi < D) {
            const float d = Ij - Ic[i];
            const float k = ex2_approx(fmaf(d * d, cI, s_lw[dyi * D + dxi]));
            ks[i] += k;
            s[i].x = fmaf(k, yj.x, s[i].x);
            s[i].y = fmaf(k, yj.y, s[i].y);
            s[i].z = fmaf(k, yj.z, s[i].z);
            s[i].w = fmaf(k, yj.w, s[i].w);
          }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < RT; ++i) {
      const int gy = y0 + ly0 + i, gx = x0 + lane;
      if (gy < H && gx < W) {
        const float4 yc = sY[(ly0 + i + R) * HW_ + lane + R];
        // analytic OOB part of sum k (F10)
        const int nx = min(gx + R, W - 1) - max(gx - R, 0) + 1;
        const int ny = min(gy + R, H - 1) - max(gy - R, 0) + 1;
        const int noob = D * D - nx * ny;
        float kk = ks[i];
        if (noob > 0) {
          const float e = -((float)gx * gx + (float)gy * gy) * inv2sxy2 - Ic[i] * Ic[i] * inv2srgb2;
          kk += (float)noob * weight * expf(e);
        }
        acc[0] += kk;
        acc[1] += s[i].x * yc.x + s[i].y * yc.y + s[i].z * yc.z + s[i].w * yc.w;
        if (gprobs) {
          float* gp = gprobs + n * C4 * HW + (long long)gy * W + gx;
          gp[0] = gscale * s[i].x; gp[HW] = gscale * s[i].y; gp[2 * HW] = gscale * s[i].z; gp[3 * HW] = gscale * s[i].w;
        }
      }
    }
  }
  __shared__ double res[2];
  if (block_reduce_final<2, 32 * WARPS>(acc, partials, ticket, res)) {
    if (threadIdx.x == 0) {
      out[0] = (float)((res[0] - res[1]) * (double)inv_denom);
      out[1] = (float)res[0];   // kernels.sum() (for diagnostics / tests)
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K9: Mumford-Shah as written in the reference (utils/losses.py:275-309, image <-> prediction roles
// swapped, F11):  level = sum_{n,k} sum_px (p_k - c_nk)^2 I,  c_nk = sum(p_k I)/sum(I);
// tv = sum|d_h p| + sum|d_w p|.   Expanded: sum (p-c)^2 I = sum p^2 I - (sum p I)^2 / sum I.
// grid = (chunks, N); per block 10 partial sums: A_k = sum p_k^2 I, B_k = sum p_k I (k<4), S = sum I, TV.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) ms_fwd_kernel(
    const float* __restrict__ image, const float* __restrict__ probs, int H, int W,
    float* partials, unsigned* ticket, float* out /*[1]*/, float* cent /*[N][4]*/, int N) {
  const int n = blockIdx.y;
  const long long HW = (long long)H * W;
  const float* I = image + n * HW;
  const float* P = probs + n * C4 * HW;
  float acc[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) acc[k] = 0.f;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < HW; i += (long long)gridDim.x * TPB) {
    const int y = (int)(i / W), x = (int)(i - (long long)y * W);
    const float iv = I[i];
    acc[8] += iv;
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      const float p = P[c * HW + i];
      acc[c] += p * p * iv;
      acc[4 + c] += p * iv;
      if (y + 1 < H) acc[9] += fabsf(P[c * HW + i + W] - p);
      if (x + 1 < W) acc[9] += fabsf(P[c * HW + i + 1] - p);
    }
  }
  // block-level partial -> partials[(n*gridDim.x + bx)*10 + k]; last block of the whole grid finalises
  __shared__ float s_w[TPB / 32][10];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    float r = warp_sum(acc[k]);
    if (lane == 0) s_w[warp][k] = r;
  }
  __syncthreads();
  if (threadIdx.x < 10) {
    float r = 0.f;
    for (int w = 0; w < TPB / 32; ++w) r += s_w[w][threadIdx.x];
    partials[((size_t)n * gridDim.x + blockIdx.x) * 10 + threadIdx.x] = r;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x * gridDim.y - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // finalize: one warp per sample (strided), fixed order, double accumulation
  __shared__ double s_loss[TPB / 32];
  double wl = 0.0;
  for (int nn = warp; nn < N; nn += TPB / 32) {
    double a[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) a[k] = 0.0;
    for (int b = lane; b < (int)gridDim.x; b += 32)
#pragma unroll
      for (int k = 0; k < 10; ++k) a[k] += (double)__ldcg(&partials[((size_t)nn * gridDim.x + b) * 10 + k]);
#pragma unroll
    for (int k = 0; k < 10; ++k)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a[k] += __shfl_xor_sync(0xffffffffu, a[k], o);
    if (lane == 0) {
      double l = a[9];
      for (int c = 0; c < C4; ++c) {
        const double cen = a[4 + c] / a[8];
        cent[nn * C4 + c] = (float)cen;
        l += a[c] - a[4 + c] * cen;
      }
      wl += l;
    }
  }
  if (lane == 0) s_loss[warp] = wl;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < TPB / 32; ++w) t += s_loss[w];
    out[0] = (float)t;
    *ticket = 0u;
  }
}

// d/dp_k = 2 (p_k - c_nk) I   (the centroid's own derivative cancels: sum (p-c) I = 0)
//        + sign(p - p_up) - sign(p_down - p) + sign(p - p_left) - sign(p_right - p)
__global__ void __launch_bounds__(TPB) ms_bwd_kernel(
    const float* __restrict__ image, const float* __restrict__ probs, const float* __restrict__ cent,
    int N, int H, int W, float scale, int accumulate, float* __restrict__ gprobs) {
  const long long HW = (long long)H * W, total = (long long)N * C4 * HW;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const long long nc = i / HW, o = i - nc * HW;
    const int n = (int)(nc / C4);
    const int y = (int)(o / W), x = (int)(o - (long long)y * W);
    const float p = probs[i];
    float g = 2.f * (p - cent[nc]) * image[n * HW + o];
    auto sgn = [](float v) { return (v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f); };
    if (y > 0) g += sgn(p - probs[i - W]);
    if (y + 1 < H) g -= sgn(probs[i + W] - p);
    if (x > 0) g += sgn(p - probs[i - 1]);
    if (x + 1 < W) g -= sgn(probs[i + 1] - p);
    g *= scale;
    gprobs[i] = accumulate ? gprobs[i] + g : g;
  }
}

// ------------------------------------------------------------------------------------------------
// K10: dynamically mixed pseudo labels + (partial) Dice.
//   pseudo = argmax_c(beta*p1 + (1-beta)*p2)   (train_weakly_supervised_segmentation_pCE_ours_proposed.py:117-120)
//   pDLoss (utils/losses.py:195-232) per class:  1 - (2*I+eps)/(Z+Y+eps),  I = sum s*t*M, Y = sum t*M, Z = sum s^2*M
//   with M[h,w] = sum_n mask[n,h,w] -- the [N,1,H,W] x [N,H,W] broadcast in the reference (losses.py:209-211,
//   219-220,229) multiplies every pixel by the batch-summed ignore mask at that location.
// The rounding of the mix follows torch: two fp32 multiplies and one fp32 add, no FMA contraction.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) mix_argmax_kernel(
    const float* __restrict__ p1, const float* __restrict__ p2, float beta, float omb, const float* __restrict__ beta_ptr,
    int HW, long long npix, uint8_t* __restrict__ out) {
  if (beta_ptr) { beta = beta_ptr[0]; omb = beta_ptr[1]; }     // device-side {beta, 1-beta}: graph replays follow the host RNG
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < npix; i += (long long)gridDim.x * TPB) {
    const long long n = i / HW, o = i - n * HW;
    const float* a = p1 + n * C4 * (long long)HW + o;
    const float* b = p2 ? p2 + n * C4 * (long long)HW + o : nullptr;
    float best = -INFINITY;
    int arg = 0;
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      float v = b ? __fadd_rn(__fmul_rn(beta, a[(long long)c * HW]), __fmul_rn(omb, b[(long long)c * HW])) : a[(long long)c * HW];
      if (v > best) { best = v; arg = c; }   // first maximum wins, as torch.argmax
    }
    out[i] = (uint8_t)arg;
  }
}

// msum[h,w] = number of samples whose target at (h,w) is not ignore_index
__global__ void __launch_bounds__(TPB) mask_count_kernel(const uint8_t* __restrict__ target, int N, int HW, int ignore_index,
                                                         float* __restrict__ msum) {
  for (int o = blockIdx.x * TPB + threadIdx.x; o < HW; o += gridDim.x * TPB) {
    int c = 0;
    for (int n = 0; n < N; ++n) c += (target[(long long)n * HW + o] != ignore_index);
    msum[o] = (float)c;
  }
}

__global__ void __launch_bounds__(TPB) pdice_fwd_kernel(
    const float* __restrict__ probs, const uint8_t* __restrict__ target, const float* __restrict__ msum, float mconst,
    int HW, long long npix, float* partials, unsigned* ticket, float* out /*[1 + 12]*/) {
  float acc[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) acc[k] = 0.f;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < npix; i += (long long)gridDim.x * TPB) {
    const long long n = i / HW, o = i - n * HW;
    const float m = msum ? msum[o] : mconst;
    const int t = target[i];
    const float* p = probs + n * C4 * (long long)HW + o;
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      const float s = p[(long long)c * HW];
      const float tt = (t == c) ? 1.f : 0.f;
      acc[c] += s * tt * m;        // I
      acc[4 + c] += tt * m;        // Y
      acc[8 + c] += s * s * m;     // Z
    }
  }
  __shared__ double res[12];
  if (block_reduce_final<12, TPB>(acc, partials, ticket, res)) {
    if (threadIdx.x == 0) {
      double loss = 0.0;
      for (int c = 0; c < C4; ++c) {
        loss += 1.0 - (2.0 * res[c] + 1e-5) / (res[8 + c] + res[4 + c] + 1e-5);
        out[1 + c] = (float)res[c]; out[5 + c] = (float)res[4 + c]; out[9 + c] = (float)res[8 + c];
      }
      out[0] = (float)(loss / C4);
    }
  }
}

// d loss / d s_c(px) = -(1/C) * [ 2 t M (Z+Y+eps) - (2I+eps) 2 s M ] / (Z+Y+eps)^2
__global__ void __launch_bounds__(TPB) pdice_bwd_kernel(
    const float* __restrict__ probs, const uint8_t* __restrict__ target, const float* __restrict__ msum, float mconst,
    const float* __restrict__ sums /*out of fwd: [1+12]*/, int HW, long long npix, float scale, int accumulate,
    float* __restrict__ gprobs) {
  float a[C4], b[C4];
#pragma unroll
  for (int c = 0; c < C4; ++c) {
    const double den = (double)sums[9 + c] + (double)sums[5 + c] + 1e-5;
    const double num = 2.0 * (double)sums[1 + c] + 1e-5;
    a[c] = (float)(-(double)scale / C4 * 2.0 / den);          // coefficient of t*M
    b[c] = (float)((double)scale / C4 * 2.0 * num / (den * den));  // coefficient of s*M
  }
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < npix; i += (long long)gridDim.x * TPB) {
    const long long n = i / HW, o = i - n * HW;
    const float m = msum ? msum[o] : mconst;
    const int t = target[i];
    const long long base = n * C4 * (long long)HW + o;
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      const float s = probs[base + (long long)c * HW];
      const float g = (a[c] * ((t == c) ? 1.f : 0.f) + b[c] * s) * m;
      float* gp = gprobs + base + (long long)c * HW;
      *gp = accumulate ? *gp + g : g;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K11: TV / contour-length loss (train_weakly_supervised_pCE_TV_2D.py:58-65):
//   mn = minpool3(p), contour = relu(maxpool3(mn) - mn), loss = mean(contour); pools see only in-bounds
//   pixels (max_pool2d pads with -inf).  Backward routes like autograd: +g to the argmin of the window
//   that attains the max, -g to the argmin of the centre window (first extremum in row-major scan order).
//   The atomics add +-1 (integer counts, exact in fp32 in any order) and tv_scale_kernel multiplies by g
//   afterwards: adding +-g directly rounds partial sums such as 3g, so the result would depend on the
//   order of the atomics, run to run, and contributions that cancel could leave a residue instead of 0.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float minpool_at(const float* P, int H, int W, int y, int x, int* arg) {
  float best = INFINITY;
  int a = -1;
  for (int dy = -1; dy <= 1; ++dy)
    for (int dx = -1; dx <= 1; ++dx) {
      int yy = y + dy, xx = x + dx;
      if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
      float v = P[yy * W + xx];
      if (a < 0 || v < best) { best = v; a = yy * W + xx; }
    }
  if (arg) *arg = a;
  return best;
}

__global__ void __launch_bounds__(TPB) tv_kernel(
    const float* __restrict__ probs, int planes, int H, int W, float* __restrict__ gcount,
    float* partials, unsigned* ticket, float* out) {
  const long long HW = (long long)H * W, total = (long long)planes * HW;
  float acc[1] = {0.f};
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const long long pl = i / HW;
    const int o = (int)(i - pl * HW), y = o / W, x = o - y * W;
    const float* P = probs + pl * HW;
    int argc;
    const float mc = minpool_at(P, H, W, y, x, &argc);
    float mx = -INFINITY;
    int argm = -1, argmx = -1;
    for (int dy = -1; dy <= 1; ++dy)
      for (int dx = -1; dx <= 1; ++dx) {
        int yy = y + dy, xx = x + dx;
        if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
        int a;
        float v = minpool_at(P, H, W, yy, xx, &a);
        if (v > mx || argmx < 0) { mx = v; argm = a; argmx = yy * W + xx; }
      }
    const float c = mx - mc;
    if (c > 0.f) {
      acc[0] += c;
      if (gcount) {
        atomicAdd(gcount + pl * HW + argm, 1.f);
        atomicAdd(gcount + pl * HW + argc, -1.f);
      }
    }
  }
  __shared__ double res[1];
  if (block_reduce_final<1, TPB>(acc, partials, ticket, res)) {
    if (threadIdx.x == 0) out[0] = (float)(res[0] / (double)total);
  }
}

__global__ void __launch_bounds__(TPB) tv_scale_kernel(float* __restrict__ g, long long total, float gscale /*go/numel*/) {
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) g[i] *= gscale;
}

// ------------------------------------------------------------------------------------------------
// K13: uncertainty-aware mean-teacher consistency (train_uncertainty_aware_mean_teacher_2D.py:164-188):
//   p_bar  = mean_t softmax(mc_logits[t])                         (T stochastic teacher passes, :164-174)
//   unc    = -sum_c p_bar log(p_bar + 1e-6)                       (:175-176)
//   mask   = unc < threshold                                      (:184-186)
//   dist_c = (softmax(student)_c - softmax(teacher)_c)^2          (utils/losses.py:65-82, softmax_mse_loss)
//   loss   = sum(mask * dist) / (2 * sum(mask) + 1e-16)           (:187-188)
// mc_logits is the [T*B,4,H,W] buffer the script fills with T/2 teacher calls on the twice-repeated batch:
// row (2*B*i + r) holds pass t = 2i + r/B of sample r % B.
// fwd: one pass, emits the mask (u8) and {sum masked dist, mask count, loss}; bwd: d loss/d student logits.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void softmax4(const float (&x)[C4], float (&p)[C4]) {
  const float m = fmaxf(fmaxf(x[0], x[1]), fmaxf(x[2], x[3]));
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < C4; ++c) { p[c] = expf(x[c] - m); s += p[c]; }
  const float inv = 1.f / s;
#pragma unroll
  for (int c = 0; c < C4; ++c) p[c] *= inv;
}

__global__ void __launch_bounds__(TPB) uamt_consistency_fwd_kernel(
    const float* __restrict__ student, const float* __restrict__ teacher, const float* __restrict__ mc, int T, int B, int HW,
    const float* __restrict__ threshold_ptr, float threshold, uint8_t* __restrict__ mask, float* partials, unsigned* ticket,
    float* out /*[3]: sum, count, loss*/) {
  const float thr = threshold_ptr ? *threshold_ptr : threshold;
  float acc[2] = {0.f, 0.f};
  const long long npix = (long long)B * HW;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < npix; i += (long long)gridDim.x * TPB) {
    const long long b = i / HW, o = i - b * HW;
    float pbar[C4] = {0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < T; ++t) {
      const long long row = (long long)(t >> 1) * 2 * B + (long long)(t & 1) * B + b;
      float x[C4], p[C4];
#pragma unroll
      for (int c = 0; c < C4; ++c) x[c] = mc[(row * C4 + c) * HW + o];
      softmax4(x, p);
#pragma unroll
      for (int c = 0; c < C4; ++c) pbar[c] += p[c];
    }
    float unc = 0.f;
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      const float q = pbar[c] / (float)T;
      unc -= q * logf(q + 1e-6f);
    }
    const bool on = unc < thr;
    mask[i] = on ? 1 : 0;
    if (on) {
      float xs[C4], xt[C4], ps[C4], pt[C4];
#pragma unroll
      for (int c = 0; c < C4; ++c) { xs[c] = student[(b * C4 + c) * HW + o]; xt[c] = teacher[(b * C4 + c) * HW + o]; }
      softmax4(xs, ps);
      softmax4(xt, pt);
      float d = 0.f;
#pragma unroll
      for (int c = 0; c < C4; ++c) d += (ps[c] - pt[c]) * (ps[c] - pt[c]);
      acc[0] += d;
      acc[1] += 1.f;
    }
  }
  __shared__ double res[2];
  if (block_reduce_final<2, TPB>(acc, partials, ticket, res)) {
    if (threadIdx.x == 0) {
      out[0] = (float)res[0];
      out[1] = (float)res[1];
      out[2] = (float)(res[0] / (2.0 * res[1] + 1e-16));
    }
  }
}

// d (w * loss) / d student logits = softmax-Jacobian applied to g_c = w * 2 * mask * (ps_c - pt_c) / (2*count + 1e-16)
__global__ void __launch_bounds__(TPB) uamt_consistency_bwd_kernel(
    const float* __restrict__ student, const float* __restrict__ teacher, const uint8_t* __restrict__ mask,
    const float* __restrict__ stats, const float* __restrict__ weight_ptr, float weight, int B, int HW,
    float* __restrict__ dlogits) {
  const float w = (weight_ptr ? *weight_ptr : weight) * 2.f / (2.f * stats[1] + 1e-16f);
  const long long npix = (long long)B * HW;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < npix; i += (long long)gridDim.x * TPB) {
    const long long b = i / HW, o = i - b * HW;
    float d[C4] = {0.f, 0.f, 0.f, 0.f};
    if (mask[i]) {
      float xs[C4], xt[C4], ps[C4], pt[C4], g[C4];
#pragma unroll
      for (int c = 0; c < C4; ++c) { xs[c] = student[(b * C4 + c) * HW + o]; xt[c] = teacher[(b * C4 + c) * HW + o]; }
      softmax4(xs, ps);
      softmax4(xt, pt);
      float dot = 0.f;
#pragma unroll
      for (int c = 0; c < C4; ++c) { g[c] = w * (ps[c] - pt[c]); dot += g[c] * ps[c]; }
#pragma unroll
      for (int c = 0; c < C4; ++c) d[c] = ps[c] * (g[c] - dot);
    }
#pragma unroll
    for (int c = 0; c < C4; ++c) dlogits[(b * C4 + c) * HW + o] = d[c];
  }
}

// x + clamp(sigma * N(0,1), -c, c): torch.clamp(torch.randn_like(x) * 0.1, -0.2, 0.2) + x (:147-149,167-169) with the
// counter RNG (Box-Muller); `reps` stacks the batch (x.repeat(reps,1,1,1)).
__global__ void __launch_bounds__(TPB) add_clamped_noise_kernel(const float* __restrict__ x, long long n, int reps, float sigma,
                                                                float clampv, unsigned long long seed,
                                                                const unsigned long long* seed_ptr, float* __restrict__ out) {
  if (seed_ptr) seed += *seed_ptr;
  const long long total = n * reps;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const float u1 = fmaxf(wsl_uniform(seed, (unsigned long long)(2 * i)), 1e-7f);
    const float u2 = wsl_uniform(seed, (unsigned long long)(2 * i + 1));
    const float z = sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
    out[i] = x[i % n] + fminf(fmaxf(z * sigma, -clampv), clampv);
  }
}

// ------------------------------------------------------------------------------------------------
// Validation path (val_2D.py:18-50, SURVEY 8(f) rank 1): scipy.ndimage.zoom(order=0) of every slice to the
// network size and of the label map back, and per-class overlap counts for Dice, on the GPU for a whole volume.
// zoom(order=0) as SciPy computes it: coordinate cc = o * (in-1)/(out-1) in double, index floor(cc + 0.5),
// and -- mode='constant' -- a coordinate that rounding pushes past in-1 reads cval = 0 (this does happen for the
// last row/column of some sizes; reproduced because the reference's predictions contain it).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int zoom0_index(int o, int n_in, int n_out, bool& oob) {
  const double scale = (n_out > 1) ? (double)(n_in - 1) / (double)(n_out - 1) : 0.0;
  const double cc = (double)o * scale;
  oob = (cc < 0.0) || (cc > (double)(n_in - 1));
  int i = (int)floor(cc + 0.5);
  return i < 0 ? 0 : (i > n_in - 1 ? n_in - 1 : i);
}

template <typename T>
__global__ void __launch_bounds__(TPB) zoom_nearest_kernel(const T* __restrict__ src, int S, int h, int w, int H, int W,
                                                           T* __restrict__ dst) {
  const long long total = (long long)S * H * W;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const int x = (int)(i % W), y = (int)((i / W) % H);
    const long long s = i / ((long long)W * H);
    bool oy, ox;
    const int iy = zoom0_index(y, h, H, oy), ix = zoom0_index(x, w, W, ox);
    dst[i] = (oy || ox) ? (T)0 : src[(s * h + iy) * w + ix];
  }
}

// counts[c] = {|pred==c & gt==c|, |pred==c|, |gt==c|} for c = 1..classes-1 (medpy.metric.binary.dc inputs)
__global__ void __launch_bounds__(TPB) overlap_counts_kernel(const uint8_t* __restrict__ pred, const uint8_t* __restrict__ gt,
                                                             long long n, int classes, unsigned long long* __restrict__ counts) {
  __shared__ unsigned int s_c[16 * 3];
  for (int i = threadIdx.x; i < 48; i += TPB) s_c[i] = 0;
  __syncthreads();
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < n; i += (long long)gridDim.x * TPB) {
    const int p = pred[i], g = gt[i];
    if (p > 0 && p < classes) atomicAdd(&s_c[p * 3 + 1], 1u);
    if (g > 0 && g < classes) atomicAdd(&s_c[g * 3 + 2], 1u);
    if (p == g && p > 0 && p < classes) atomicAdd(&s_c[p * 3 + 0], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < classes * 3; i += TPB)
    if (s_c[i]) atomicAdd(&counts[i], (unsigned long long)s_c[i]);
}

// ------------------------------------------------------------------------------------------------
// Entropy minimisation: losses.entropy_loss(p, C) = mean_px(-sum_c p log(p + 1e-6)) / log(C)  (utils/losses.py:30-36,
// train_weakly_supervised_pCE_Entropy_Mini_2D.py:99-102).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) entropy_fwd_kernel(const float* __restrict__ probs, long long total, float inv_norm,
                                                          float* partials, unsigned* ticket, float* out) {
  float acc[1] = {0.f};
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const float p = probs[i];
    acc[0] -= p * logf(p + 1e-6f);
  }
  __shared__ double res[1];
  if (block_reduce_final<1, TPB>(acc, partials, ticket, res)) {
    if (threadIdx.x == 0) out[0] = (float)(res[0] * (double)inv_norm);
  }
}

__global__ void __launch_bounds__(TPB) entropy_bwd_kernel(const float* __restrict__ probs, long long total, float scale,
                                                          int accumulate, float* __restrict__ gprobs) {
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const float p = probs[i];
    const float g = -scale * (logf(p + 1e-6f) + p / (p + 1e-6f));
    gprobs[i] = accumulate ? gprobs[i] + g : g;
  }
}

// ------------------------------------------------------------------------------------------------
// Inter / intra class variance (train_weakly_supervised_pCE_Inter&Intra_Class_2D.py:30-36,114):
//   v = img * p_c;  intra = mean_{n,c} std_{hw}(v)  (unbiased);  inter = mean_n std_c(mean_{hw}(v))  (unbiased over C)
//   loss = inter - intra.   fwd: per-(n,c) sums S1 = sum v, S2 = sum v^2 (grid = (chunks, N)), finalised by the last
//   block into stats[n][c] = {mean, std} + stats_n[n] = {mean over classes, std over classes}; bwd is elementwise.
// A zero standard deviation yields a zero gradient, as torch's std backward does (it masks result == 0).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) variance_fwd_kernel(const float* __restrict__ image, const float* __restrict__ probs, int N,
                                                           long long HW, float* partials, unsigned* ticket, float* out /*[3]*/,
                                                           float* stats /*[N*4*2 + N*2]*/) {
  const int n = blockIdx.y;
  float acc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = 0.f;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < HW; i += (long long)gridDim.x * TPB) {
    const float iv = image[n * HW + i];
#pragma unroll
    for (int c = 0; c < C4; ++c) {
      const float v = iv * probs[(n * C4 + c) * HW + i];
      acc[c] += v;
      acc[4 + c] = fmaf(v, v, acc[4 + c]);
    }
  }
  __shared__ float s_w[TPB / 32][8];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float r = warp_sum(acc[k]);
    if (lane == 0) s_w[warp][k] = r;
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    float r = 0.f;
    for (int w = 0; w < TPB / 32; ++w) r += s_w[w][threadIdx.x];
    partials[((size_t)n * gridDim.x + blockIdx.x) * 8 + threadIdx.x] = r;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x * gridDim.y - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  __shared__ double s_intra[TPB / 32], s_inter[TPB / 32];
  double w_intra = 0.0, w_inter = 0.0;
  const double M = (double)HW;
  for (int nn = warp; nn < N; nn += TPB / 32) {
    double a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = 0.0;
    for (int b = lane; b < (int)gridDim.x; b += 32)
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] += (double)__ldcg(&partials[((size_t)nn * gridDim.x + b) * 8 + k]);
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a[k] += __shfl_xor_sync(0xffffffffu, a[k], o);
    if (lane == 0) {
      double mean[C4], mbar = 0.0;
      for (int c = 0; c < C4; ++c) {
        mean[c] = a[c] / M;
        double var = (a[4 + c] - a[c] * a[c] / M) / (M - 1.0);
        if (var < 0.0) var = 0.0;
        const double sd = sqrt(var);
        stats[(nn * C4 + c) * 2 + 0] = (float)mean[c];
        stats[(nn * C4 + c) * 2 + 1] = (float)sd;
        w_intra += sd;
        mbar += mean[c];
      }
      mbar /= C4;
      double vv = 0.0;
      for (int c = 0; c < C4; ++c) vv += (mean[c] - mbar) * (mean[c] - mbar);
      const double sdn = sqrt(vv / (C4 - 1.0));
      stats[N * C4 * 2 + nn * 2 + 0] = (float)mbar;
      stats[N * C4 * 2 + nn * 2 + 1] = (float)sdn;
      w_inter += sdn;
    }
  }
  if (lane == 0) { s_intra[warp] = w_intra; s_inter[warp] = w_inter; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ia = 0.0, ie = 0.0;
    for (int w = 0; w < TPB / 32; ++w) { ia += s_intra[w]; ie += s_inter[w]; }
    ia /= (double)(N * C4);
    ie /= (double)N;
    out[0] = (float)(ie - ia);
    out[1] = (float)ie;
    out[2] = (float)ia;
    *ticket = 0u;
  }
}

__global__ void __launch_bounds__(TPB) variance_bwd_kernel(const float* __restrict__ image, const float* __restrict__ probs,
                                                           const float* __restrict__ stats, int N, long long HW, float scale,
                                                           int accumulate, float* __restrict__ gprobs) {
  const long long total = (long long)N * C4 * HW;
  const float M = (float)HW;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const long long nc = i / HW, o = i - nc * HW;
    const int n = (int)(nc / C4);
    const float iv = image[n * HW + o];
    const float v = iv * probs[i];
    const float mean = stats[nc * 2], sd = stats[nc * 2 + 1];
    const float mbar = stats[N * C4 * 2 + n * 2], sdn = stats[N * C4 * 2 + n * 2 + 1];
    float g = 0.f;
    if (sdn > 0.f) g += (mean - mbar) / ((C4 - 1.f) * sdn * M * (float)N);                 // + d inter / d v
    if (sd > 0.f) g -= (v - mean) / ((M - 1.f) * sd * (float)(N * C4));                    // - d intra / d v
    g *= scale * iv;
    gprobs[i] = accumulate ? gprobs[i] + g : g;
  }
}

// torch.rot90(x, k, [2, 3]) for square maps (train_weakly_supervised_ustm_2D.py:124-125,150): k=1: out[i][j] = in[j][S-1-i];
// k=2: out[i][j] = in[S-1-i][S-1-j]; k=3: out[i][j] = in[S-1-j][i].  accumulate: dst += rot(src).
__global__ void __launch_bounds__(TPB) rot90_kernel(const float* __restrict__ src, long long planes, int S, int k, int accumulate,
                                                    float* __restrict__ dst) {
  const long long total = planes * S * S;
  for (long long t = blockIdx.x * (long long)TPB + threadIdx.x; t < total; t += (long long)gridDim.x * TPB) {
    const int j = (int)(t % S), i = (int)((t / S) % S);
    const long long pl = t / ((long long)S * S);
    int si, sj;
    switch (k & 3) {
      case 1: si = j; sj = S - 1 - i; break;
      case 2: si = S - 1 - i; sj = S - 1 - j; break;
      case 3: si = S - 1 - j; sj = i; break;
      default: si = i; sj = j; break;
    }
    const float v = src[(pl * S + si) * S + sj];
    dst[t] = accumulate ? dst[t] + v : v;
  }
}

// update_ema_variables (train_weakly_supervised_ustm_2D.py:61-65): ema = alpha*ema + (1-alpha)*param over a flat buffer
__global__ void __launch_bounds__(TPB) ema_update_kernel(float* __restrict__ ema, const float* __restrict__ param, long long n, float alpha) {
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < n; i += (long long)gridDim.x * TPB)
    ema[i] = ema[i] * alpha + (1.f - alpha) * param[i];
}

// torch.nn.functional.interpolate(x, size) with the default mode='nearest' on fp32 [planes, h, w] maps (Decoder_DS heads,
// networks/unet.py:177,181,185): src index = min(floor(dst * (in / out)), in - 1) with the scale in float, as ATen computes it.
__device__ __forceinline__ int nearest_src(int dst, float scale, int in_size) {
  const int s = (int)floorf((float)dst * scale);
  return s < in_size - 1 ? s : in_size - 1;
}

__global__ void __launch_bounds__(TPB) nearest_resize_fwd_kernel(const float* __restrict__ src, long long planes, int h, int w, int H,
                                                                 int W, float* __restrict__ dst) {
  const float sy = (float)h / (float)H, sx = (float)w / (float)W;
  const long long total = planes * H * W;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const int x = (int)(i % W), y = (int)((i / W) % H);
    const long long pl = i / ((long long)W * H);
    dst[i] = src[(pl * h + nearest_src(y, sy, h)) * w + nearest_src(x, sx, w)];
  }
}

// its transpose (gather form, deterministic): every source pixel sums the destination pixels that read it
__global__ void __launch_bounds__(TPB) nearest_resize_bwd_kernel(const float* __restrict__ gdst, long long planes, int h, int w, int H,
                                                                 int W, float* __restrict__ gsrc) {
  const float sy = (float)h / (float)H, sx = (float)w / (float)W;
  const long long total = planes * h * w;
  for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < total; i += (long long)gridDim.x * TPB) {
    const int xs = (int)(i % w), ys = (int)((i / w) % h);
    const long long pl = i / ((long long)w * h);
    // candidate destination range: dst*scale in [src, src+1)  (one extra on both sides for float rounding, then tested exactly)
    int y0 = (int)((float)ys / sy) - 1, y1 = (int)((float)(ys + 1) / sy) + 1;
    int x0 = (int)((float)xs / sx) - 1, x1 = (int)((float)(xs + 1) / sx) + 1;
    y0 = y0 < 0 ? 0 : y0; x0 = x0 < 0 ? 0 : x0; y1 = y1 > H - 1 ? H - 1 : y1; x1 = x1 > W - 1 ? W - 1 : x1;
    float acc = 0.f;
    for (int y = y0; y <= y1; ++y) {
      if (nearest_src(y, sy, h) != ys) continue;
      for (int x = x0; x <= x1; ++x)
        if (nearest_src(x, sx, w) == xs) acc += gdst[(pl * H + y) * W + x];
    }
    gsrc[i] = acc;
  }
}

inline int grid_for(long long work_items, int per_block) {
  long long b = (work_items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  if (b > 148 * 8) b = 148 * 8;   // multiple of the SM count; grid-stride loops cover the rest
  return (int)b;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
WSL_API int wsl_softmax_pce_fwd(const float* logits, const uint8_t* label, float* probs, int N, int C, int H, int W,
                                int ignore_index, float* out2, float* ws, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_softmax_pce_fwd: C must be 4 (got %d)", C);
  WSL_REQUIRE(((long long)H * W) % 4 == 0, "wsl_softmax_pce_fwd: H*W must be a multiple of 4");
  const long long nq = (long long)N * H * W / 4;
  const int grid = grid_for(nq, TPB);
  softmax_pce_fwd_kernel<<<grid, TPB, 0, stream>>>(logits, label, probs, H * W, nq, ignore_index, ws + 64,
                                                   reinterpret_cast<unsigned*>(ws), out2);
  return wsl_check_launch("softmax_pce_fwd");
}

WSL_API int wsl_head_bwd(const float* probs, const uint8_t* label, const float* ce_stats, const float* grad_out,
                         float w_ce, const float* gprobs, float gprobs_scale, int N, int C, int H, int W,
                         int ignore_index, float* dlogits, void* dlogits_nhwc16, int dtype16, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_head_bwd: C must be 4 (got %d)", C);
  WSL_REQUIRE(((long long)H * W) % 4 == 0, "wsl_head_bwd: H*W must be a multiple of 4");
  const long long nq = (long long)N * H * W / 4;
  head_bwd_kernel<<<grid_for(nq, TPB), TPB, 0, stream>>>(probs, label, ce_stats, grad_out, w_ce, gprobs, gprobs_scale,
                                                         H * W, nq, ignore_index, dlogits, (__nv_bfloat16*)dlogits_nhwc16, dtype16);
  return wsl_check_launch("head_bwd");
}

WSL_API int wsl_gatedcrf_fwd(const float* probs, const float* image, float* gprobs, int N, int C, int H, int W,
                             int radius, float sigma_xy, float sigma_rgb, float weight, float* out2, float* ws,
                             cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_gatedcrf_fwd: C must be 4 (got %d)", C);
  WSL_REQUIRE(radius == 5, "wsl_gatedcrf_fwd: fused path is compiled for radius 5 (got %d)", radius);
  constexpr int R = 5, RT = 8, WARPS = 4;
  constexpr int TW = 32, TH = RT * WARPS;
  const int tx = (W + TW - 1) / TW, ty = (H + TH - 1) / TH;
  const long long ntiles = (long long)N * tx * ty;
  int grid = (int)(ntiles < WSL_MAX_PARTIAL_BLOCKS ? ntiles : 148 * 12);
  const size_t smem = (((TH + 2 * R) * (TW + 2 * R) + 3) & ~3) * sizeof(float) + (size_t)(TH + 2 * R) * (TW + 2 * R) * sizeof(float4);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(gatedcrf_kernel<R, RT, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    attr_set = true;
  }
  const double denom = (double)N * H * W;
  gatedcrf_kernel<R, RT, WARPS><<<grid, 32 * WARPS, smem, stream>>>(
      probs, image, gprobs, N, H, W, 0.5f / (sigma_xy * sigma_xy), 0.5f / (sigma_rgb * sigma_rgb), weight,
      (float)(-2.0 / denom), tx, ty, ws + 64, reinterpret_cast<unsigned*>(ws), out2, (float)(1.0 / denom));
  return wsl_check_launch("gatedcrf_fwd");
}

WSL_API int wsl_mumford_shah_fwd(const float* image, const float* probs, int N, int C, int H, int W, float* out1,
                                 float* centroids, float* ws, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_mumford_shah_fwd: C must be 4 (got %d)", C);
  int chunks = (int)(((long long)H * W + TPB * 4 - 1) / (TPB * 4));
  if (chunks > 64) chunks = 64;
  WSL_REQUIRE((long long)chunks * N * 10 <= (long long)WSL_MAX_PARTIAL_BLOCKS * 32, "wsl_mumford_shah_fwd: batch too large for workspace");
  ms_fwd_kernel<<<dim3(chunks, N), TPB, 0, stream>>>(image, probs, H, W, ws + 64, reinterpret_cast<unsigned*>(ws), out1,
                                                     centroids, N);
  return wsl_check_launch("mumford_shah_fwd");
}

WSL_API int wsl_mumford_shah_bwd(const float* image, const float* probs, const float* centroids, int N, int C, int H,
                                 int W, float scale, int accumulate, float* gprobs, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_mumford_shah_bwd: C must be 4 (got %d)", C);
  ms_bwd_kernel<<<grid_for((long long)N * C * H * W, TPB), TPB, 0, stream>>>(image, probs, centroids, N, H, W, scale,
                                                                             accumulate, gprobs);
  return wsl_check_launch("mumford_shah_bwd");
}

WSL_API int wsl_mix_argmax(const float* p1, const float* p2, float beta, float one_minus_beta, const float* beta_ptr, int N, int C,
                           int H, int W, uint8_t* out, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_mix_argmax: C must be 4 (got %d)", C);
  const long long npix = (long long)N * H * W;
  mix_argmax_kernel<<<grid_for(npix, TPB), TPB, 0, stream>>>(p1, p2, beta, one_minus_beta, beta_ptr, H * W, npix, out);
  return wsl_check_launch("mix_argmax");
}

WSL_API int wsl_mask_count(const uint8_t* target, int N, int H, int W, int ignore_index, float* msum, cudaStream_t stream) {
  mask_count_kernel<<<grid_for((long long)H * W, TPB), TPB, 0, stream>>>(target, N, H * W, ignore_index, msum);
  return wsl_check_launch("mask_count");
}

WSL_API int wsl_pdice_fwd(const float* probs, const uint8_t* target, const float* msum, float mconst, int N, int C, int H,
                          int W, float* out13, float* ws, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_pdice_fwd: C must be 4 (got %d)", C);
  const long long npix = (long long)N * H * W;
  pdice_fwd_kernel<<<grid_for(npix, TPB), TPB, 0, stream>>>(probs, target, msum, mconst, H * W, npix, ws + 64,
                                                            reinterpret_cast<unsigned*>(ws), out13);
  return wsl_check_launch("pdice_fwd");
}

WSL_API int wsl_pdice_bwd(const float* probs, const uint8_t* target, const float* msum, float mconst, const float* sums13,
                          int N, int C, int H, int W, float scale, int accumulate, float* gprobs, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_pdice_bwd: C must be 4 (got %d)", C);
  const long long npix = (long long)N * H * W;
  pdice_bwd_kernel<<<grid_for(npix, TPB), TPB, 0, stream>>>(probs, target, msum, mconst, sums13, H * W, npix, scale,
                                                            accumulate, gprobs);
  return wsl_check_launch("pdice_bwd");
}

WSL_API int wsl_tv_loss(const float* probs, int planes, int H, int W, float grad_scale, float* gprobs_zeroed, float* out1,
                        float* ws, cudaStream_t stream) {
  const long long total = (long long)planes * H * W;
  tv_kernel<<<grid_for(total, TPB), TPB, 0, stream>>>(probs, planes, H, W, gprobs_zeroed, ws + 64, reinterpret_cast<unsigned*>(ws),
                                                      out1);
  if (gprobs_zeroed != nullptr)
    tv_scale_kernel<<<grid_for(total, TPB * 4), TPB, 0, stream>>>(gprobs_zeroed, total, grad_scale / (float)total);
  return wsl_check_launch("tv_loss");
}

WSL_API int wsl_uamt_consistency_fwd(const float* student, const float* teacher, const float* mc_logits, int T, int B, int C,
                                     int H, int W, const float* threshold_ptr, float threshold, uint8_t* mask, float* out3,
                                     float* ws, cudaStream_t stream) {
  WSL_REQUIRE(C == C4 && T >= 2 && T % 2 == 0, "wsl_uamt_consistency_fwd: C must be 4 and T even (got C=%d, T=%d)", C, T);
  const long long npix = (long long)B * H * W;
  uamt_consistency_fwd_kernel<<<grid_for(npix, TPB), TPB, 0, stream>>>(student, teacher, mc_logits, T, B, H * W, threshold_ptr,
                                                                       threshold, mask, ws + 64, reinterpret_cast<unsigned*>(ws), out3);
  return wsl_check_launch("uamt_consistency_fwd");
}

WSL_API int wsl_uamt_consistency_bwd(const float* student, const float* teacher, const uint8_t* mask, const float* stats3,
                                     const float* weight_ptr, float weight, int B, int C, int H, int W, float* dlogits,
                                     cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_uamt_consistency_bwd: C must be 4 (got %d)", C);
  const long long npix = (long long)B * H * W;
  uamt_consistency_bwd_kernel<<<grid_for(npix, TPB), TPB, 0, stream>>>(student, teacher, mask, stats3, weight_ptr, weight, B,
                                                                       H * W, dlogits);
  return wsl_check_launch("uamt_consistency_bwd");
}

WSL_API int wsl_add_clamped_noise(const float* x, long long n, int reps, float sigma, float clamp, unsigned long long seed,
                                  const unsigned long long* seed_ptr, float* out, cudaStream_t stream) {
  add_clamped_noise_kernel<<<grid_for(n * reps, TPB), TPB, 0, stream>>>(x, n, reps, sigma, clamp, seed, seed_ptr, out);
  return wsl_check_launch("add_clamped_noise");
}

WSL_API int wsl_zoom_nearest(const void* src, int is_u8, int S, int h, int w, int H, int W, void* dst, cudaStream_t stream) {
  const long long total = (long long)S * H * W;
  if (is_u8) zoom_nearest_kernel<uint8_t><<<grid_for(total, TPB), TPB, 0, stream>>>((const uint8_t*)src, S, h, w, H, W, (uint8_t*)dst);
  else zoom_nearest_kernel<float><<<grid_for(total, TPB), TPB, 0, stream>>>((const float*)src, S, h, w, H, W, (float*)dst);
  return wsl_check_launch("zoom_nearest");
}

WSL_API int wsl_overlap_counts(const uint8_t* pred, const uint8_t* gt, long long n, int classes, unsigned long long* counts_zeroed,
                               cudaStream_t stream) {
  WSL_REQUIRE(classes >= 2 && classes <= 16, "wsl_overlap_counts: 2..16 classes (got %d)", classes);
  overlap_counts_kernel<<<grid_for(n, TPB * 4), TPB, 0, stream>>>(pred, gt, n, classes, counts_zeroed);
  return wsl_check_launch("overlap_counts");
}

WSL_API int wsl_entropy_fwd(const float* probs, int N, int C, int H, int W, float* out1, float* ws, cudaStream_t stream) {
  const long long total = (long long)N * C * H * W;
  const float inv_norm = (float)(1.0 / ((double)N * H * W * log((double)C)));
  entropy_fwd_kernel<<<grid_for(total, TPB * 4), TPB, 0, stream>>>(probs, total, inv_norm, ws + 64, reinterpret_cast<unsigned*>(ws), out1);
  return wsl_check_launch("entropy_fwd");
}

WSL_API int wsl_entropy_bwd(const float* probs, int N, int C, int H, int W, float scale, int accumulate, float* gprobs,
                            cudaStream_t stream) {
  const long long total = (long long)N * C * H * W;
  const float sc = (float)((double)scale / ((double)N * H * W * log((double)C)));
  entropy_bwd_kernel<<<grid_for(total, TPB * 4), TPB, 0, stream>>>(probs, total, sc, accumulate, gprobs);
  return wsl_check_launch("entropy_bwd");
}

WSL_API int wsl_class_variance_fwd(const float* image, const float* probs, int N, int C, int H, int W, float* out3, float* stats,
                                   float* ws, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_class_variance_fwd: C must be 4 (got %d)", C);
  int chunks = (int)(((long long)H * W + TPB * 4 - 1) / (TPB * 4));
  if (chunks > 64) chunks = 64;
  WSL_REQUIRE((long long)chunks * N * 8 + 64 <= WSL_WS_FLOATS, "wsl_class_variance_fwd: batch too large for the workspace");
  variance_fwd_kernel<<<dim3(chunks, N), TPB, 0, stream>>>(image, probs, N, (long long)H * W, ws + 64, reinterpret_cast<unsigned*>(ws),
                                                           out3, stats);
  return wsl_check_launch("class_variance_fwd");
}

WSL_API int wsl_class_variance_bwd(const float* image, const float* probs, const float* stats, int N, int C, int H, int W,
                                   float scale, int accumulate, float* gprobs, cudaStream_t stream) {
  WSL_REQUIRE(C == C4, "wsl_class_variance_bwd: C must be 4 (got %d)", C);
  variance_bwd_kernel<<<grid_for((long long)N * C * H * W, TPB * 2), TPB, 0, stream>>>(image, probs, stats, N, (long long)H * W, scale,
                                                                                      accumulate, gprobs);
  return wsl_check_launch("class_variance_bwd");
}

WSL_API int wsl_rot90(const float* src, long long planes, int S, int k, int accumulate, float* dst, cudaStream_t stream) {
  WSL_REQUIRE(src != dst, "wsl_rot90: in-place rotation is not supported");
  rot90_kernel<<<grid_for(planes * S * S, TPB * 2), TPB, 0, stream>>>(src, planes, S, k, accumulate, dst);
  return wsl_check_launch("rot90");
}

WSL_API int wsl_ema_update(float* ema, const float* param, long long n, float alpha, cudaStream_t stream) {
  ema_update_kernel<<<grid_for(n, TPB * 2), TPB, 0, stream>>>(ema, param, n, alpha);
  return wsl_check_launch("ema_update");
}

WSL_API int wsl_nearest_resize_fwd(const float* src, long long planes, int h, int w, int H, int W, float* dst, cudaStream_t stream) {
  nearest_resize_fwd_kernel<<<grid_for(planes * H * W, TPB * 2), TPB, 0, stream>>>(src, planes, h, w, H, W, dst);
  return wsl_check_launch("nearest_resize_fwd");
}

WSL_API int wsl_nearest_resize_bwd(const float* gdst, long long planes, int h, int w, int H, int W, float* gsrc, cudaStream_t stream) {
  nearest_resize_bwd_kernel<<<grid_for(planes * h * w, TPB), TPB, 0, stream>>>(gdst, planes, h, w, H, W, gsrc);
  return wsl_check_launch("nearest_resize_bwd");
}
