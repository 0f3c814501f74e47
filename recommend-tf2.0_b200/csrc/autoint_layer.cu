// K6 — the AutoInt interacting layer, whole layer in ONE launch per direction.
//
// ctr.layers.modules.MultiHeadAttention.call on a self-attention input X (B, F, dm)
// (src/ctr/layers/modules.py:255-270, 211-220, 235-240, 281-283, 316-323):
//   Q, K, V = act(X Wq), act(X Wk), act(X Wv)         no bias, activation on all three
//   per head h:  P = softmax(Q_h K_h^T * scale)       scale = sqrt(hs) in the reference form
//                O_h = P V_h                          no mask
//   out = O                       (use_res = False)
//   out = relu(O + act(X W0))     (use_res = True)
// The layer is 354 kFLOP on 7.5 KB per sample (SURVEY §8d): fp32-FMA-bound, so one CTA keeps a
// sample's X, Q, K, V, residual and the score matrices in shared memory and nothing but X and
// out touches HBM.  The reference lowers it to 4 tensordots, 2 transposes, 2 batched GEMMs and
// a softmax, each an HBM round trip.
//
// Mapping (128 threads): projections — warp m <-> matrix {Q,K,V,R}, lane <-> output column,
// the thread's weight column lives in registers for the whole launch, X rows come as 128-bit
// broadcast loads; attention — one thread per (head, query row), scores staged in shared
// memory, fp32 softmax with the row maximum subtracted (same formula as the oracle).
// Backward recomputes Q/K/V/R/P (cheaper than 20 KB per sample of HBM), then
//   phase A (thread per query row)  dP = dO V^T, dS = P (dP - sum_j P dP) scale, dQ = dS K
//   phase B (thread per key row)    dV = P^T dO, dK = dS^T Q        (no atomics: fixed order)
//   phase C                         dX = sum_m (d_m . act'(M_m)) W_m^T
//   phase D                         dW_m += X^T (d_m . act') accumulated in REGISTERS over the
//                                   CTA's samples (fixed grid, fixed order); the per-CTA
//                                   partials are summed in CTA order by a second tiny kernel,
// so the weight gradients are reproducible bit for bit.
#include "rtf_common.cuh"

namespace rtf {

enum { AI_ACT_NONE = 0, AI_ACT_RELU = 1, AI_ACT_SIGMOID = 2, AI_ACT_TANH = 3 };
constexpr int AI_THREADS = 128;
constexpr int AI_MAXF = 64;

__device__ __forceinline__ float ai_act(int act, float z) {
  switch (act) {
    case AI_ACT_RELU: return fmaxf(z, 0.f);
    case AI_ACT_SIGMOID: return 1.f / (1.f + expf(-z));
    case AI_ACT_TANH: return tanhf(z);
    default: return z;
  }
}
// derivative expressed through the activation's OUTPUT y
__device__ __forceinline__ float ai_dact(int act, float y) {
  switch (act) {
    case AI_ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case AI_ACT_SIGMOID: return y * (1.f - y);
    case AI_ACT_TANH: return 1.f - y * y;
    default: return 1.f;
  }
}

struct AiParams {
  const float* x;    // (B, F, DM)
  const float* w[4]; // Wq, Wk, Wv, W0 (DM, HS) row-major; w[3] null without residual
  float* out;        // fwd (B, F, HS)
  const float* outr; // bwd: forward output (relu mask of the residual form)
  const float* gout; // bwd (B, F, HS)
  float* gx;         // bwd (B, F, DM)
  float* partial;    // bwd [gridDim.x][4][DM][HS]
  long long B;
  int F, H, act, use_res;
  float scale;
};

// shared-memory layout (floats), sized by the actual field count F:
//   Xs [F][DM] | Q K V R, each [F][HS] (stride kMat = F*HS) | (bwd: dO [F][HS]) |
//   P [H][F][F|1] (| bwd: dS, same shape); score rows have an ODD stride: a thread walks its own
//   row, so lanes (different rows) must land in different banks (stride 40 was 8-way conflicted).

// projections of one sample: M_m[r][c] = act(sum_k X[r][k] W_m[k][c]) for the thread's (m, c)
template <int DM, int HS>
__device__ __forceinline__ void ai_project(const float* __restrict__ Xs, float* __restrict__ Ms,
                                           const float (&wreg)[(HS + 31) / 32][DM], int F, int act,
                                           int m, int lane, bool live) {
  if (!live) return;
  const int kMat = F * HS;
#pragma unroll
  for (int cc = 0; cc < (HS + 31) / 32; ++cc) {
    const int c = lane + 32 * cc;
    if (c >= HS) continue;
    float* dst = Ms + m * kMat + c;
    for (int r0 = 0; r0 < F; r0 += 4) {   // 4 independent accumulation chains
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k4 = 0; k4 < DM / 4; ++k4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int r = min(r0 + u, F - 1);
          const float4 xv = *reinterpret_cast<const float4*>(Xs + r * DM + 4 * k4);
          acc[u] = fmaf(xv.x, wreg[cc][4 * k4 + 0], acc[u]);
          acc[u] = fmaf(xv.y, wreg[cc][4 * k4 + 1], acc[u]);
          acc[u] = fmaf(xv.z, wreg[cc][4 * k4 + 2], acc[u]);
          acc[u] = fmaf(xv.w, wreg[cc][4 * k4 + 3], acc[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (r0 + u < F) dst[(r0 + u) * HS] = ai_act(act, acc[u]);
    }
  }
}

// softmax row of query (h, i): P[h][i][:] (normalised) into Ps; returns nothing
template <int DM, int HS, int HSZ>
__device__ __forceinline__ void ai_scores(const float* __restrict__ Ms, float* __restrict__ Ps,
                                          int F, int h, int i, float scale) {
  const int kMat = F * HS, kS = F | 1;
  const float* Q = Ms;
  const float* K = Ms + kMat;
  float q[HSZ];
#pragma unroll
  for (int d4 = 0; d4 < HSZ / 4; ++d4) {
    const float4 t = *reinterpret_cast<const float4*>(Q + i * HS + h * HSZ + 4 * d4);
    q[4 * d4] = t.x; q[4 * d4 + 1] = t.y; q[4 * d4 + 2] = t.z; q[4 * d4 + 3] = t.w;
  }
  float* prow = Ps + (h * F + i) * kS;
  float mx = -INFINITY;
  for (int j0 = 0; j0 < F; j0 += 4) {     // 4 independent dot products
    float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int d4 = 0; d4 < HSZ / 4; ++d4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = min(j0 + u, F - 1);
        const float4 kv = *reinterpret_cast<const float4*>(K + j * HS + h * HSZ + 4 * d4);
        s4[u] = fmaf(q[4 * d4], kv.x, s4[u]);
        s4[u] = fmaf(q[4 * d4 + 1], kv.y, s4[u]);
        s4[u] = fmaf(q[4 * d4 + 2], kv.z, s4[u]);
        s4[u] = fmaf(q[4 * d4 + 3], kv.w, s4[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (j0 + u < F) {
        const float s = s4[u] * scale;
        prow[j0 + u] = s;
        mx = fmaxf(mx, s);
      }
  }
  float sum = 0.f;
  for (int j = 0; j < F; ++j) {
    const float e = expf(prow[j] - mx);
    prow[j] = e;
    sum += e;
  }
  const float inv = 1.f / sum;
  for (int j = 0; j < F; ++j) prow[j] *= inv;
}

template <int DM, int HS>
__device__ __forceinline__ void ai_load_weights(const AiParams& P, float (&wreg)[(HS + 31) / 32][DM],
                                                int m, int lane, bool live) {
#pragma unroll
  for (int cc = 0; cc < (HS + 31) / 32; ++cc)
#pragma unroll
    for (int k = 0; k < DM; ++k) {
      const int c = lane + 32 * cc;
      wreg[cc][k] = (live && c < HS) ? __ldg(P.w[m] + k * HS + c) : 0.f;
    }
}

template <int DM, int HS>
__device__ __forceinline__ void ai_load_x(const float* __restrict__ src, float* __restrict__ Xs, int n) {
  for (int e = threadIdx.x * 4; e < n; e += AI_THREADS * 4)
    *reinterpret_cast<float4*>(Xs + e) = ldg_nc_f4(src + e);
}

// ---- forward, packed FMAs (sm_100 FFMA2: two fp32 FMAs per issue slot) -----------------------
// Scalar FFMA, as in ai_project / ai_scores above, is bound by the FMA pipe's issue rate (one FFMA
// per 2 cycles and scheduler).  Here every contraction is arranged so that BOTH halves of a packed
// FMA are useful and come out of the loads already paired:
//   projections: X is staged TRANSPOSED (Xt[k][row]), one 128-bit broadcast load gives 4 rows of
//                column k = two row pairs; {w,w} pairs live in registers for the whole launch;
//   Q K^T:       K is written transposed by its projection (Kt[col][key]); a thread owns a query
//                row, keeps its scores in REGISTERS (FP/2 float2) and adds {q_d,q_d} x {K_j,K_j+1};
//   P V:         pairs over the head dimension come straight from V's rows, {p,p} is one move.
// FP = compile-time bound on the field count (multiple of 4); softmax as in ai_scores.
template <int DM, int HS, int HSZ, int FP>
__global__ void __launch_bounds__(AI_THREADS, FP <= 40 ? 4 : 2)
autoint_fwd2_kernel(const __grid_constant__ AiParams P) {
  extern __shared__ __align__(16) float sm[];
  constexpr int NC = (HS + 31) / 32;
  const int F = P.F, H = P.H;
  float* Xt = sm;                 // [DM][FP]   X transposed
  float* Qt = Xt + DM * FP;       // [HS][FP]   Q transposed (lanes = query rows read it conflict-free)
  float* Kt = Qt + FP * HS;       // [HS][FP]   K transposed
  float* Vs = Kt + HS * FP;       // [FP][HS]
  float* Rs = Vs + FP * HS;       // [FP][HS]
  const int lane = threadIdx.x & 31, m = threadIdx.x >> 5;
  const bool live = m < 3 || P.use_res;
  float2 ww[NC][DM];              // {w,w} of this thread's weight column(s)
#pragma unroll
  for (int cc = 0; cc < NC; ++cc)
#pragma unroll
    for (int k = 0; k < DM; ++k) {
      const int c = lane + 32 * cc;
      const float w = (live && c < HS) ? __ldg(P.w[m] + k * HS + c) : 0.f;
      ww[cc][k] = make_float2(w, w);
    }
  for (int e = threadIdx.x; e < DM * FP; e += AI_THREADS) Xt[e] = 0.f;   // pad rows stay zero
  __syncthreads();
  for (long long b = blockIdx.x; b < P.B; b += gridDim.x) {
    const float* xg = P.x + b * F * DM;
    for (int e = threadIdx.x; e < F * DM; e += AI_THREADS) {
      const int r = e / DM, k = e - r * DM;
      Xt[k * FP + r] = __ldg(xg + e);
    }
    __syncthreads();
    // ---- projections: thread (matrix m, column c), rows in pairs
    if (live) {
#pragma unroll
      for (int cc = 0; cc < NC; ++cc) {
        const int c = lane + 32 * cc;
        if (c >= HS) continue;
        float* dst = m == 2 ? Vs : Rs;
#pragma unroll 2
        for (int r0 = 0; r0 < FP; r0 += 4) {
          float2 a0 = make_float2(0.f, 0.f), a1 = make_float2(0.f, 0.f);
#pragma unroll
          for (int k = 0; k < DM; ++k) {
            const float4 x4 = *reinterpret_cast<const float4*>(Xt + k * FP + r0);
            a0 = __ffma2_rn(make_float2(x4.x, x4.y), ww[cc][k], a0);
            a1 = __ffma2_rn(make_float2(x4.z, x4.w), ww[cc][k], a1);
          }
          const float v[4] = {ai_act(P.act, a0.x), ai_act(P.act, a0.y), ai_act(P.act, a1.x),
                              ai_act(P.act, a1.y)};
          if (m <= 1) {   // Q and K leave transposed
            *reinterpret_cast<float4*>((m == 0 ? Qt : Kt) + c * FP + r0) =
                make_float4(v[0], v[1], v[2], v[3]);
          } else {
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (r0 + u < F) dst[(r0 + u) * HS + c] = v[u];
          }
        }
      }
    }
    __syncthreads();
    // ---- attention: thread per (head, query row); scores in registers
    for (int p = threadIdx.x; p < H * F; p += AI_THREADS) {
      const int h = p / F, i = p - h * F;
      float2 s2[FP / 2];
#pragma unroll
      for (int j = 0; j < FP / 2; ++j) s2[j] = make_float2(0.f, 0.f);
#pragma unroll
      for (int d = 0; d < HSZ; ++d) {
        const float q = Qt[(h * HSZ + d) * FP + i];
        const float2 qq = make_float2(q, q);
        const float* kt = Kt + (h * HSZ + d) * FP;
#pragma unroll
        for (int j4 = 0; j4 < FP / 4; ++j4) {
          const float4 k4 = *reinterpret_cast<const float4*>(kt + 4 * j4);
          s2[2 * j4] = __ffma2_rn(qq, make_float2(k4.x, k4.y), s2[2 * j4]);
          s2[2 * j4 + 1] = __ffma2_rn(qq, make_float2(k4.z, k4.w), s2[2 * j4 + 1]);
        }
      }
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < FP / 2; ++j) {
        s2[j].x = 2 * j < F ? s2[j].x * P.scale : -INFINITY;
        s2[j].y = 2 * j + 1 < F ? s2[j].y * P.scale : -INFINITY;
        mx = fmaxf(mx, fmaxf(s2[j].x, s2[j].y));
      }
      float sum = 0.f;
#pragma unroll
      for (int j = 0; j < FP / 2; ++j) {
        s2[j].x = 2 * j < F ? expf(s2[j].x - mx) : 0.f;
        s2[j].y = 2 * j + 1 < F ? expf(s2[j].y - mx) : 0.f;
        sum += s2[j].x + s2[j].y;
      }
      const float inv = 1.f / sum;
      float2 o2[HSZ / 2];
#pragma unroll
      for (int d = 0; d < HSZ / 2; ++d) o2[d] = make_float2(0.f, 0.f);
      const float* V = Vs + h * HSZ;
#pragma unroll
      for (int j = 0; j < FP; ++j) {
        if (j < F) {
          const float pj = ((j & 1) ? s2[j >> 1].y : s2[j >> 1].x) * inv;
          const float2 pp = make_float2(pj, pj);
#pragma unroll
          for (int d4 = 0; d4 < HSZ / 4; ++d4) {
            const float4 vv = *reinterpret_cast<const float4*>(V + j * HS + 4 * d4);
            o2[2 * d4] = __ffma2_rn(pp, make_float2(vv.x, vv.y), o2[2 * d4]);
            o2[2 * d4 + 1] = __ffma2_rn(pp, make_float2(vv.z, vv.w), o2[2 * d4 + 1]);
          }
        }
      }
      float* dst = P.out + (b * F + i) * HS + h * HSZ;
      const float* R = Rs + i * HS + h * HSZ;
#pragma unroll
      for (int d4 = 0; d4 < HSZ / 4; ++d4) {
        float4 v = make_float4(o2[2 * d4].x, o2[2 * d4].y, o2[2 * d4 + 1].x, o2[2 * d4 + 1].y);
        if (P.use_res) {
          const float4 r = *reinterpret_cast<const float4*>(R + 4 * d4);
          v.x = fmaxf(v.x + r.x, 0.f);
          v.y = fmaxf(v.y + r.y, 0.f);
          v.z = fmaxf(v.z + r.z, 0.f);
          v.w = fmaxf(v.w + r.w, 0.f);
        }
        *reinterpret_cast<float4*>(dst + 4 * d4) = v;
      }
    }
    __syncthreads();  // Xt / Qt / Kt / V / R are overwritten by the next sample
  }
}

template <int DM, int HS, int HSZ>
__global__ void __launch_bounds__(AI_THREADS, 2)
autoint_bwd_kernel(const __grid_constant__ AiParams P) {
  extern __shared__ __align__(16) float sm[];
  constexpr int NC = (HS + 31) / 32;
  const int F = P.F, H = P.H;
  const int kMat = F * HS, kS = F | 1;
  float* Xs = sm;                        // [F][DM]
  float* Ms = Xs + F * DM;               // Q | K | V | R  ->  dQpre | dKpre | dVpre | dRpre
  float* dO = Ms + 4 * kMat;             // [F][HS] gradient entering the attention output
  float* Ps = dO + kMat;                 // [H][F][kS] probabilities
  float* dSs = Ps + H * F * kS;          // [H][F][kS] dS
  const int lane = threadIdx.x & 31, m = threadIdx.x >> 5;
  const bool live = m < 3 || P.use_res;
  float wreg[NC][DM];
  ai_load_weights<DM, HS>(P, wreg, m, lane, live);
  float gw[NC][DM];   // dW_m[:, c] of this thread, accumulated over the CTA's samples
#pragma unroll
  for (int cc = 0; cc < NC; ++cc)
#pragma unroll
    for (int k = 0; k < DM; ++k) gw[cc][k] = 0.f;

  for (long long b = blockIdx.x; b < P.B; b += gridDim.x) {
    ai_load_x<DM, HS>(P.x + b * F * DM, Xs, F * DM);
    // dO = gout (. relu mask of the forward output in the residual form)
    for (int e = threadIdx.x * 4; e < F * HS; e += AI_THREADS * 4) {
      float4 g = ldg_nc_f4(P.gout + b * F * HS + e);
      if (P.use_res) {
        const float4 y = ldg_nc_f4(P.outr + b * F * HS + e);
        g.x = y.x > 0.f ? g.x : 0.f;
        g.y = y.y > 0.f ? g.y : 0.f;
        g.z = y.z > 0.f ? g.z : 0.f;
        g.w = y.w > 0.f ? g.w : 0.f;
      }
      *reinterpret_cast<float4*>(dO + e) = g;
    }
    __syncthreads();
    ai_project<DM, HS>(Xs, Ms, wreg, F, P.act, m, lane, live);
    __syncthreads();
    // ---- phase A: thread per (head, query row)
    float dq[HSZ];
    int myh = -1, myi = -1;
    for (int p = threadIdx.x; p < H * F; p += AI_THREADS) {   // H*F <= 128: one trip per thread
      const int h = p / F, i = p - h * F;
      myh = h; myi = i;
      ai_scores<DM, HS, HSZ>(Ms, Ps, F, h, i, P.scale);
      const float* prow = Ps + (h * F + i) * kS;
      float* dsrow = dSs + (h * F + i) * kS;
      const float* V = Ms + 2 * kMat + h * HSZ;
      const float* K = Ms + kMat + h * HSZ;
      float go[HSZ];
#pragma unroll
      for (int d4 = 0; d4 < HSZ / 4; ++d4) {
        const float4 t = *reinterpret_cast<const float4*>(dO + i * HS + h * HSZ + 4 * d4);
        go[4 * d4] = t.x; go[4 * d4 + 1] = t.y; go[4 * d4 + 2] = t.z; go[4 * d4 + 3] = t.w;
      }
      float delta = 0.f;
      for (int j0 = 0; j0 < F; j0 += 4) {
        float dp4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int d4 = 0; d4 < HSZ / 4; ++d4) {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int j = min(j0 + u, F - 1);
            const float4 vv = *reinterpret_cast<const float4*>(V + j * HS + 4 * d4);
            dp4[u] = fmaf(go[4 * d4], vv.x, dp4[u]);
            dp4[u] = fmaf(go[4 * d4 + 1], vv.y, dp4[u]);
            dp4[u] = fmaf(go[4 * d4 + 2], vv.z, dp4[u]);
            dp4[u] = fmaf(go[4 * d4 + 3], vv.w, dp4[u]);
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (j0 + u < F) {
            dsrow[j0 + u] = dp4[u];
            delta = fmaf(prow[j0 + u], dp4[u], delta);
          }
      }
#pragma unroll
      for (int d = 0; d < HSZ; ++d) dq[d] = 0.f;
      for (int j = 0; j < F; ++j) {
        const float ds = prow[j] * (dsrow[j] - delta) * P.scale;
        dsrow[j] = ds;
        const float4* kr = reinterpret_cast<const float4*>(K + j * HS);
#pragma unroll
        for (int d4 = 0; d4 < HSZ / 4; ++d4) {
          const float4 kv = kr[d4];
          dq[4 * d4] = fmaf(ds, kv.x, dq[4 * d4]);
          dq[4 * d4 + 1] = fmaf(ds, kv.y, dq[4 * d4 + 1]);
          dq[4 * d4 + 2] = fmaf(ds, kv.z, dq[4 * d4 + 2]);
          dq[4 * d4 + 3] = fmaf(ds, kv.w, dq[4 * d4 + 3]);
        }
      }
    }
    __syncthreads();
    // ---- phase B: the same thread as key row j = myi of head myh
    float dk[HSZ], dv[HSZ];
    if (myh >= 0) {
      const int h = myh, j = myi;
      const float* Q = Ms + h * HSZ;
#pragma unroll
      for (int d = 0; d < HSZ; ++d) dk[d] = dv[d] = 0.f;
      for (int i = 0; i < F; ++i) {
        const float pij = Ps[(h * F + i) * kS + j];
        const float dsij = dSs[(h * F + i) * kS + j];
        const float4* gr = reinterpret_cast<const float4*>(dO + i * HS + h * HSZ);
        const float4* qr = reinterpret_cast<const float4*>(Q + i * HS);
#pragma unroll
        for (int d4 = 0; d4 < HSZ / 4; ++d4) {
          const float4 gv = gr[d4], qv = qr[d4];
          dv[4 * d4] = fmaf(pij, gv.x, dv[4 * d4]);
          dv[4 * d4 + 1] = fmaf(pij, gv.y, dv[4 * d4 + 1]);
          dv[4 * d4 + 2] = fmaf(pij, gv.z, dv[4 * d4 + 2]);
          dv[4 * d4 + 3] = fmaf(pij, gv.w, dv[4 * d4 + 3]);
          dk[4 * d4] = fmaf(dsij, qv.x, dk[4 * d4]);
          dk[4 * d4 + 1] = fmaf(dsij, qv.y, dk[4 * d4 + 1]);
          dk[4 * d4 + 2] = fmaf(dsij, qv.z, dk[4 * d4 + 2]);
          dk[4 * d4 + 3] = fmaf(dsij, qv.w, dk[4 * d4 + 3]);
        }
      }
    }
    __syncthreads();  // every read of Q / K / V / P / dS is done: overwrite in place with d.act'
    if (myh >= 0) {
      float* Qr = Ms + myi * HS + myh * HSZ;
      float* Kr = Ms + kMat + myi * HS + myh * HSZ;
      float* Vr = Ms + 2 * kMat + myi * HS + myh * HSZ;
#pragma unroll
      for (int d = 0; d < HSZ; ++d) {
        Qr[d] = dq[d] * ai_dact(P.act, Qr[d]);
        Kr[d] = dk[d] * ai_dact(P.act, Kr[d]);
        Vr[d] = dv[d] * ai_dact(P.act, Vr[d]);
      }
    }
    if (P.use_res) {
      float* R = Ms + 3 * kMat;
      for (int e = threadIdx.x; e < F * HS; e += AI_THREADS) R[e] = dO[e] * ai_dact(P.act, R[e]);
    }
    __syncthreads();
    // ---- phase C: dX[r][k] = sum_m sum_c d_m[r][c] W_m[k][c]   (thread: k = tid % DM, rows strided)
    {
      constexpr int RG = AI_THREADS / DM;          // row groups
      const int k = threadIdx.x % DM, rg = threadIdx.x / DM;
      const int nm = P.use_res ? 4 : 3;
      for (int r0 = rg; r0 < F; r0 += RG * 4) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int mm = 0; mm < nm; ++mm) {
          const float* wrow = P.w[mm] + k * HS;    // L1/L2-resident (16 KB of weights)
          const float* dm_ = Ms + mm * kMat;
#pragma unroll 2
          for (int c4 = 0; c4 < HS / 4; ++c4) {
            const float4 wv = __ldg(reinterpret_cast<const float4*>(wrow) + c4);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int r = r0 + u * RG;
              if (r < F) {
                const float4 dvv = *reinterpret_cast<const float4*>(dm_ + r * HS + 4 * c4);
                acc[u] = fmaf(dvv.x, wv.x, acc[u]);
                acc[u] = fmaf(dvv.y, wv.y, acc[u]);
                acc[u] = fmaf(dvv.z, wv.z, acc[u]);
                acc[u] = fmaf(dvv.w, wv.w, acc[u]);
              }
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int r = r0 + u * RG;
          if (r < F) P.gx[(b * F + r) * DM + k] = acc[u];
        }
      }
    }
    // ---- phase D: dW_m[k][c] += sum_r X[r][k] d_m[r][c]   (registers, fixed sample order)
    if (live) {
#pragma unroll
      for (int cc = 0; cc < NC; ++cc) {
        const int c = lane + 32 * cc;
        if (c >= HS) continue;
        const float* dcol = Ms + m * kMat + c;
        for (int r = 0; r < F; ++r) {
          const float dv_ = dcol[r * HS];
          const float4* xr = reinterpret_cast<const float4*>(Xs + r * DM);
#pragma unroll
          for (int k4 = 0; k4 < DM / 4; ++k4) {
            const float4 xv = xr[k4];
            gw[cc][4 * k4] = fmaf(xv.x, dv_, gw[cc][4 * k4]);
            gw[cc][4 * k4 + 1] = fmaf(xv.y, dv_, gw[cc][4 * k4 + 1]);
            gw[cc][4 * k4 + 2] = fmaf(xv.z, dv_, gw[cc][4 * k4 + 2]);
            gw[cc][4 * k4 + 3] = fmaf(xv.w, dv_, gw[cc][4 * k4 + 3]);
          }
        }
      }
    }
    __syncthreads();  // Xs / Ms / dO are overwritten by the next sample
  }
  // per-CTA partial weight gradients
  float* part = P.partial + (long long)blockIdx.x * 4 * DM * HS + m * DM * HS;
#pragma unroll
  for (int cc = 0; cc < NC; ++cc) {
    const int c = lane + 32 * cc;
    if (c >= HS) continue;
#pragma unroll
    for (int k = 0; k < DM; ++k) part[k * HS + c] = gw[cc][k];
  }
}

// gW[e] = sum over CTAs (ascending) of partial[cta][e]
__global__ void __launch_bounds__(256)
autoint_dw_reduce(const float* __restrict__ partial, int ncta, int n, float* __restrict__ gW) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float acc = 0.f;
  int c = 0;
  for (; c + 16 <= ncta; c += 16) {     // 16 loads in flight, added in the same (ascending) order
    float t[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) t[u] = partial[(long long)(c + u) * n + e];
#pragma unroll
    for (int u = 0; u < 16; ++u) acc = __fadd_rn(acc, t[u]);
  }
  for (; c < ncta; ++c) acc = __fadd_rn(acc, partial[(long long)c * n + e]);
  gW[e] = acc;
}

static size_t ai_round16(size_t nfloats) { return (nfloats + 3) / 4 * 4 * sizeof(float); }
template <int DM, int HS>
static size_t ai_bwd_smem(int F, int H) {
  return ai_round16((size_t)F * DM + 5 * (size_t)F * HS + 2 * (size_t)H * F * (F | 1));
}

static int ai_grid(long long B, int per_sm) {
  long long g = (long long)kNumSMs * per_sm;
  return (int)(B < g ? B : g);
}

template <int DM, int HS, int HSZ, int FP>
static int ai_launch_fwd2(const AiParams& P, cudaStream_t st) {
  const size_t smem = ai_round16((size_t)DM * FP + 4 * (size_t)FP * HS);
  if (smem > 227 * 1024) return RTF_E_RANGE;
  cudaError_t e = cudaFuncSetAttribute(autoint_fwd2_kernel<DM, HS, HSZ, FP>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  int per_sm = (int)((227 * 1024) / (smem + 1024));
  const int cap = FP <= 40 ? 4 : 2;
  if (per_sm > cap) per_sm = cap;
  if (per_sm < 1) per_sm = 1;
  autoint_fwd2_kernel<DM, HS, HSZ, FP><<<ai_grid(P.B, per_sm), AI_THREADS, smem, st>>>(P);
  RTF_CHECK_LAUNCH();
  return 0;
}

template <int DM, int HS, int HSZ>
static int ai_launch_fwd(const AiParams& P, cudaStream_t st) {
  if (P.F <= 16) return ai_launch_fwd2<DM, HS, HSZ, 16>(P, st);
  if (P.F <= 40) return ai_launch_fwd2<DM, HS, HSZ, 40>(P, st);
  return ai_launch_fwd2<DM, HS, HSZ, 64>(P, st);
}

}  // namespace rtf

using namespace rtf;

static int ai_bwd_ctas(int64_t B) {
  const long long g = (long long)kNumSMs * 2;
  return (int)(B < g ? (B > 0 ? B : 1) : g);
}

// supported (dm, H*hs, hs) combinations of the fused layer; anything else: RTF_E_RANGE and the
// host composes the layer from the projection GEMMs + rtf_attn_* instead
#define AI_DISPATCH(CALL)                                                     \
  if (dm == 16 && HS == 32 && hs == 16) { CALL(16, 32, 16); }                 \
  else if (dm == 32 && HS == 32 && hs == 16) { CALL(32, 32, 16); }            \
  else if (dm == 16 && HS == 16 && hs == 16) { CALL(16, 16, 16); }            \
  else if (dm == 16 && HS == 8 && hs == 8) { CALL(16, 8, 8); }                \
  else if (dm == 8 && HS == 16 && hs == 8) { CALL(8, 16, 8); }                \
  else if (dm == 64 && HS == 64 && hs == 32) { CALL(64, 64, 32); }            \
  else return RTF_E_RANGE;

static int ai_check(int64_t B, int F, int dm, int H, int hs, int act, const float* x,
                    const float* wq, const float* wk, const float* wv) {
  if (B < 0 || F <= 0 || dm <= 0 || H <= 0 || hs <= 0) return RTF_E_ARG;
  if (act < AI_ACT_NONE || act > AI_ACT_TANH) return RTF_E_ARG;
  if (B > 0 && (!x || !wq || !wk || !wv)) return RTF_E_ARG;
  if (F > AI_MAXF || H * F > AI_THREADS) return RTF_E_RANGE;
  if ((uintptr_t)x % 16 || (uintptr_t)wq % 16 || (uintptr_t)wk % 16 || (uintptr_t)wv % 16)
    return RTF_E_ALIGN;
  return 0;
}

extern "C" int rtf_autoint_layer_supported(int F, int dm, int H, int hs) {
  const int HS = H * hs;
  if (F <= 0 || F > AI_MAXF || H * F > AI_THREADS) return 0;
  return (dm == 16 && HS == 32 && hs == 16) || (dm == 32 && HS == 32 && hs == 16) ||
         (dm == 16 && HS == 16 && hs == 16) || (dm == 16 && HS == 8 && hs == 8) ||
         (dm == 8 && HS == 16 && hs == 8) || (dm == 64 && HS == 64 && hs == 32);
}

extern "C" int rtf_autoint_layer_workspace(int64_t B, int dm, int HS, size_t* bytes) {
  if (!bytes || B < 0 || dm <= 0 || HS <= 0) return RTF_E_ARG;
  *bytes = (size_t)ai_bwd_ctas(B) * 4 * dm * HS * sizeof(float);
  return 0;
}

extern "C" int rtf_autoint_layer_fwd(const float* d_x, int64_t B, int F, int dm, const float* d_wq,
                                     const float* d_wk, const float* d_wv, const float* d_w0, int H,
                                     int hs, int act, float scale, float* d_out, void* stream) {
  int rc = ai_check(B, F, dm, H, hs, act, d_x, d_wq, d_wk, d_wv);
  if (rc) return rc;
  if (B > 0 && !d_out) return RTF_E_ARG;
  if ((uintptr_t)d_out % 16) return RTF_E_ALIGN;
  const int HS = H * hs;
  AiParams P = {};
  P.x = d_x; P.w[0] = d_wq; P.w[1] = d_wk; P.w[2] = d_wv; P.w[3] = d_w0;
  P.out = d_out; P.B = B; P.F = F; P.H = H; P.act = act; P.use_res = d_w0 != nullptr;
  P.scale = scale;
  if (B == 0) return 0;
#define AI_FWD(DM_, HS_, HSZ_) return ai_launch_fwd<DM_, HS_, HSZ_>(P, (cudaStream_t)stream)
  AI_DISPATCH(AI_FWD)
#undef AI_FWD
}

template <int DM, int HS, int HSZ>
static int ai_launch_bwd(AiParams& P, float* d_gw, cudaStream_t st) {
  const size_t smem = ai_bwd_smem<DM, HS>(P.F, P.H);
  if (smem > 227 * 1024) return RTF_E_RANGE;
  cudaError_t e = cudaFuncSetAttribute(autoint_bwd_kernel<DM, HS, HSZ>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const int ctas = ai_bwd_ctas(P.B);
  autoint_bwd_kernel<DM, HS, HSZ><<<ctas, AI_THREADS, smem, st>>>(P);
  RTF_CHECK_LAUNCH();
  const int n = 4 * DM * HS;
  autoint_dw_reduce<<<(n + 255) / 256, 256, 0, st>>>(P.partial, ctas, n, d_gw);
  RTF_CHECK_LAUNCH();
  return 0;
}

extern "C" int rtf_autoint_layer_bwd(const float* d_x, int64_t B, int F, int dm, const float* d_wq,
                                     const float* d_wk, const float* d_wv, const float* d_w0, int H,
                                     int hs, int act, float scale, const float* d_out,
                                     const float* d_gout, float* d_gx, float* d_gw, void* d_ws,
                                     size_t ws_bytes, void* stream) {
  int rc = ai_check(B, F, dm, H, hs, act, d_x, d_wq, d_wk, d_wv);
  if (rc) return rc;
  if (B > 0 && (!d_gout || !d_gx || !d_gw || !d_ws || (d_w0 && !d_out))) return RTF_E_ARG;
  if ((uintptr_t)d_gout % 16 || (uintptr_t)d_out % 16) return RTF_E_ALIGN;
  const int HS = H * hs;
  size_t need = 0;
  rtf_autoint_layer_workspace(B, dm, HS, &need);
  if (B > 0 && ws_bytes < need) return RTF_E_WORKSPACE;
  AiParams P = {};
  P.x = d_x; P.w[0] = d_wq; P.w[1] = d_wk; P.w[2] = d_wv; P.w[3] = d_w0;
  P.outr = d_out; P.gout = d_gout; P.gx = d_gx; P.partial = (float*)d_ws;
  P.B = B; P.F = F; P.H = H; P.act = act; P.use_res = d_w0 != nullptr; P.scale = scale;
  if (B == 0) {
    cudaMemsetAsync(d_gw, 0, (size_t)4 * dm * HS * sizeof(float), (cudaStream_t)stream);
    return 0;
  }
#define AI_BWD(DM_, HS_, HSZ_) return ai_launch_bwd<DM_, HS_, HSZ_>(P, d_gw, (cudaStream_t)stream)
  AI_DISPATCH(AI_BWD)
#undef AI_BWD
}
