// Decoder window forward: CellStateEncoder + (T-1) autoregressive GRU steps in ONE persistent
// cooperative kernel.  Replaces Decoder.forward (ZEGGS/modules.py:47-162), RecurrentDecoderNormal
// (:165-185), CellStateEncoder (:230-243), vectorize_input (:677-713), devectorize_output (:716-742).
//
// Partitioning: G = H/U CTAs, CTA c owns hidden units [c*U, (c+1)*U) of layer0 / GRU0 / GRU1 and
// ceil(1131/G) rows of layer2.  Every step is 4 weight-stationary "skinny GEMM" stages separated by a
// grid barrier; each CTA streams its own pre-packed k-major weight slice (L2 resident) and the
// k-major activation vector of the previous stage:
//   S1  x_pose(t)            -> a(t) = ELU(W0p x + S0[t]),  gi0p = W_ih0[:,pose] x + S1[t]
//   S2  a(t), h0(t-1)        -> h0(t)   (GRU layer 0; r,z,n with b_hn inside r*(.))
//   S3  h0(t), h1(t-1)       -> h1(t)   (GRU layer 1)
//   S4  h1(t)                -> y(t) = W2 h1 + b2 -> de-normalise -> pose(t), root integration,
//                               x_pose(t+1) = normalise(pose(t), gaze(t+1))
// The speech/style columns of W0 / W_ih0 do not depend on the recurrence and are hoisted out of the
// time loop into one batched pre-pass (S0/S1 above).
#include "decoder_common.cuh"

namespace zeggs {

// ------------------------------------------------------------------ weight packing
// P1[c][k][r]  r in [0,4U): g=r/U (0: layer0, 1..3: W_ih0 gate g-1), unit j=c*U+r%U, k over pose cols
// P2[c][k][r]  r in [0,6U): r<3U: W_ih0[g*H+j][k] (hidden cols), else W_hh0[g*H+j][k]
// P3[c][k][r]  same with W_ih1 / W_hh1
// P4[c][tile][k][16]  W2 rows c*rpc + tile*16 + r
__global__ void pack_decoder_kernel(DecGeom g, const float* __restrict__ W0, const float* __restrict__ Wih0,
                                    const float* __restrict__ Whh0, const float* __restrict__ Wih1,
                                    const float* __restrict__ Whh1, const float* __restrict__ W2,
                                    float* __restrict__ out) {
  const size_t total = g.packed_floats();
  const int H = g.H, U = g.U, A = g.A;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    float v = 0.f;
    if (i < g.off_p2()) {
      size_t e = i;
      int r = e % (4 * U); e /= (4 * U);
      int k = e % K1P; int c = e / K1P;
      int gi = r / U, j = c * U + r % U;
      if (k < P_IN) v = (gi == 0) ? W0[(size_t)j * A + k] : Wih0[(size_t)((gi - 1) * H + j) * (A + H) + H + k];
    } else if (i < g.off_p4()) {
      const bool l1 = i >= g.off_p3();
      size_t e = i - (l1 ? g.off_p3() : g.off_p2());
      int r = e % (6 * U); e /= (6 * U);
      int k = e % H; int c = e / H;
      const bool hh = r >= 3 * U;
      int rr = hh ? r - 3 * U : r;
      int gi = rr / U, j = c * U + rr % U;
      if (!l1) v = hh ? Whh0[(size_t)(gi * H + j) * H + k] : Wih0[(size_t)(gi * H + j) * (A + H) + k];
      else     v = hh ? Whh1[(size_t)(gi * H + j) * H + k] : Wih1[(size_t)(gi * H + j) * H + k];
    } else {
      size_t e = i - g.off_p4();
      int r = e % 16; e /= 16;
      int k = e % H; e /= H;
      int tile = e % g.n4t; int c = e / g.n4t;
      int lr = tile * 16 + r;
      int n = c * g.rpc + lr;
      if (lr < g.rpc && n < P_OUT) v = W2[(size_t)n * H + k];
    }
    out[i] = v;
  }
}

// ------------------------------------------------------------------ prologue
// frame 0 of the outputs, CellStateEncoder input [x0 | style[:,0]] and x_pose(1) = vectorize(pose0, gaze[:,1])
__global__ void decoder_prologue_kernel(zeggs_decoder_fwd_args a, DecGeom g, float* cse_in, float* xp1) {
  const int b = blockIdx.x;
  const int Z = a.Z, T = a.T;
  Q4 q; q.w = a.root_rot0[b * 4 + 0]; q.x = a.root_rot0[b * 4 + 1]; q.y = a.root_rot0[b * 4 + 2]; q.z = a.root_rot0[b * 4 + 3];
  V3 p = v3(a.root_pos0[b * 3 + 0], a.root_pos0[b * 3 + 1], a.root_pos0[b * 3 + 2]);
  const int bt = b / 32, bl = b % 32;
  float* xp = xp1 + (size_t)bt * K1P * 32;
  for (int n = threadIdx.x; n < P_IN + Z; n += blockDim.x) {
    if (n < P_OUT) {
      float v = a.pose0[(size_t)b * P_OUT + n];
      a.Y[((size_t)b * T + 0) * P_OUT + n] = v;
      float xn = (v - a.in_mean[n]) / a.in_std[n];
      cse_in[(size_t)b * (P_IN + Z) + n] = xn;
      if (T > 1) xp[(size_t)n * 32 + bl] = xn;
    } else if (n < P_IN) {
      int d = n - P_OUT;
      // gaze_dir = R(root_rot)^-1 (gaze_pos - root_pos)   modules.py:696
      V3 g0 = v3(a.gaze_pos[((size_t)b * T + 0) * 3 + 0], a.gaze_pos[((size_t)b * T + 0) * 3 + 1], a.gaze_pos[((size_t)b * T + 0) * 3 + 2]);
      V3 d0 = quat_mul_vec(quat_inv(q), g0 - p);
      float v0 = d == 0 ? d0.x : (d == 1 ? d0.y : d0.z);
      cse_in[(size_t)b * (P_IN + Z) + n] = (v0 - a.in_mean[n]) / a.in_std[n];
      if (T > 1) {
        V3 g1 = v3(a.gaze_pos[((size_t)b * T + 1) * 3 + 0], a.gaze_pos[((size_t)b * T + 1) * 3 + 1], a.gaze_pos[((size_t)b * T + 1) * 3 + 2]);
        V3 d1 = quat_mul_vec(quat_inv(q), g1 - p);
        float v1 = d == 0 ? d1.x : (d == 1 ? d1.y : d1.z);
        xp[(size_t)n * 32 + bl] = (v1 - a.in_mean[n]) / a.in_std[n];
      }
    } else {
      cse_in[(size_t)b * (P_IN + Z) + n] = a.style[((size_t)b * T + 0) * Z + (n - P_IN)];
    }
  }
  if (threadIdx.x < 3) a.root_pos[((size_t)b * T) * 3 + threadIdx.x] = a.root_pos0[b * 3 + threadIdx.x];
  if (threadIdx.x < 4) a.root_rot[((size_t)b * T) * 4 + threadIdx.x] = a.root_rot0[b * 4 + threadIdx.x];
}

// initial GRU state -> H0[slot0], H1[slot0] in k-major [bt][H][32].  Per sample b the source is the CellStateEncoder output
// cse_out[B][2H] (modules.py:243) or, when h_init is set and from_state is NULL or from_state[b] != 0, the caller's h_init[2][B][H].
__global__ void cse_scatter_kernel(int B, int H, const float* __restrict__ cse_out, const float* __restrict__ h_init,
                                   const int* __restrict__ from_state, float* __restrict__ h0, float* __restrict__ h1) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * 2 * H) return;
  int b = i / (2 * H), r = i % (2 * H);
  int l = r / H, j = r % H;
  const bool carry = h_init != nullptr && (from_state == nullptr || from_state[b] != 0);
  float* dst = l == 0 ? h0 : h1;
  dst[((size_t)(b / 32) * H + j) * 32 + (b % 32)] = carry ? h_init[((size_t)l * B + b) * H + j] : cse_out[i];
}

// h0 / h1 of one time slot (k-major [bt][H][32]) -> out[2][B][H]
__global__ void state_gather_kernel(int B, int H, const float* __restrict__ h0, const float* __restrict__ h1, float* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * B * H) return;
  int l = i / (B * H), r = i % (B * H);
  int b = r / H, j = r % H;
  out[i] = (l == 0 ? h0 : h1)[((size_t)(b / 32) * H + j) * 32 + (b % 32)];
}

// S01[t][bt][n][32], n in [0,4H): n<H: b0[n] + W0[n, 1134:] . cond ; else b_ih0[n-H] + W_ih0[n-H, H+1134:] . cond
// cond = [speech[b,t,:] | style[b,t,:]].  One CTA per (t, bt, 64-row tile).
__global__ void __launch_bounds__(256) cond_precompute_kernel(zeggs_decoder_fwd_args a, DecGeom g, float* __restrict__ S01) {
  extern __shared__ float sm[];
  const int C = a.S + a.Z, H = a.H, T = a.T, A = g.A;
  float* cs = sm;              // [C][33]
  float* ws = sm + C * 33;     // [64][C+1]
  const int t = blockIdx.x, bt = blockIdx.y, n0 = blockIdx.z * 64;
  for (int i = threadIdx.x; i < 32 * C; i += blockDim.x) {
    int bl = i / C, cc = i % C;
    int b = bt * 32 + bl;
    float v = 0.f;
    if (b < a.B) v = cc < a.S ? a.speech[((size_t)b * T + t) * a.S + cc] : a.style[((size_t)b * T + t) * a.Z + (cc - a.S)];
    cs[cc * 33 + bl] = v;
  }
  for (int i = threadIdx.x; i < 64 * C; i += blockDim.x) {
    int r = i / C, cc = i % C;
    int n = n0 + r;
    float v = 0.f;
    if (n < 4 * H) v = n < H ? a.W0[(size_t)n * A + P_IN + cc] : a.W_ih0[(size_t)(n - H) * (A + H) + H + P_IN + cc];
    ws[r * (C + 1) + cc] = v;
  }
  __syncthreads();
  const int bl = threadIdx.x & 31, rw = threadIdx.x >> 5;  // 8 warps x 8 rows
  for (int rr = 0; rr < 8; ++rr) {
    int r = rw * 8 + rr, n = n0 + r;
    if (n >= 4 * H) break;
    float acc = n < H ? a.b0[n] : a.b_ih0[n - H];
    for (int cc = 0; cc < C; ++cc) acc = fmaf(ws[r * (C + 1) + cc], cs[cc * 33 + bl], acc);
    S01[(((size_t)t * g.nbt + bt) * 4 * H + n) * 32 + bl] = acc;
  }
}

// cond rows for the tc engine: R[(t*32 + b)][c] = [speech[b,t,:] | style[b,t,:]] (zero rows for b >= B)
__global__ void cond_rows_kernel(zeggs_decoder_fwd_args a, float* __restrict__ R) {
  const int C = a.S + a.Z, T = a.T;
  const size_t total = (size_t)T * 32 * C;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int cc = (int)(i % C); const size_t e = i / C;
    const int b = (int)(e & 31), t = (int)(e >> 5);
    float v = 0.f;
    if (b < a.B) v = cc < a.S ? a.speech[((size_t)b * T + t) * a.S + cc] : a.style[((size_t)b * T + t) * a.Z + (cc - a.S)];
    R[i] = v;
  }
}

// ------------------------------------------------------------------ the persistent kernel
template <int U>
__global__ void __launch_bounds__(256, 1) decoder_fwd_kernel(zeggs_decoder_fwd_args a, DecGeom g, DecWs w) {
  extern __shared__ __align__(16) float smem[];
  constexpr int RT1 = U, RT2 = (6 * U) / 4;
  float* stage = smem;                                  // 8 warps x 2 x STG_MAX
  float* red = smem + 8 * 2 * SkinnyCfg<RT2>::STG;      // [8][6U][32]
  float* gi0p = red + 8 * 6 * U * 32;                   // [nbt][3][U][32]
  float* rootv = gi0p + g.nbt * 3 * U * 32;             // [6][32]
  const int c = blockIdx.x, tid = threadIdx.x, warp = tid >> 5;
  const int H = a.H, T = a.T, nbt = g.nbt;
  float* wstage = stage + warp * 2 * SkinnyCfg<RT2>::STG;
  GridBarrier gb; gb.counter = w.bar; gb.error = w.bar + 1; gb.epoch = 0; gb.nblocks = gridDim.x;

  const float* P1 = a.packed + (size_t)c * K1P * 4 * U;
  const float* P2 = a.packed + g.off_p2() + (size_t)c * H * 6 * U;
  const float* P3 = a.packed + g.off_p3() + (size_t)c * H * 6 * U;
  const float* P4 = a.packed + g.off_p4() + (size_t)c * g.n4t * H * 16;
  const size_t actH = (size_t)nbt * H * 32;      // floats per time slot of an [nbt][H][32] buffer
  const size_t actX = (size_t)nbt * K1P * 32;

  for (int t = 1; t < T; ++t) {
    const int ts = w.save ? t : (t & 1), tp = w.save ? t - 1 : ((t - 1) & 1), tn = w.save ? t + 1 : ((t + 1) & 1);
    // ------------------------------------------------------------ stage 1
    for (int bt = 0; bt < nbt; ++bt) {
      float acc[RT1][4];
      const float* x = w.XP + ts * actX + (size_t)bt * K1P * 32;
      skinny_gemm<RT1, false>(acc, P1, x, x, K1P / 16, wstage);
      reduce_store<RT1>(acc, red);
      __syncthreads();
      for (int idx = tid; idx < U * 32; idx += 256) {
        const int u = idx >> 5, b = idx & 31, j = c * U + u;
        const float* S = w.S01 + (((size_t)t * nbt + bt) * 4 * H) * 32;
        float pre = red_sum<4 * U>(red, u, b) + S[(size_t)j * 32 + b];
        w.A[ts * actH + ((size_t)bt * H + j) * 32 + b] = elu_f(pre);
#pragma unroll
        for (int gi = 0; gi < 3; ++gi)
          gi0p[((bt * 3 + gi) * U + u) * 32 + b] = red_sum<4 * U>(red, (1 + gi) * U + u, b) + S[(size_t)(H + gi * H + j) * 32 + b];
      }
      __syncthreads();
    }
    if (!grid_sync(gb)) return;
    // ------------------------------------------------------------ stage 2 (GRU layer 0)
    for (int bt = 0; bt < nbt; ++bt) {
      float acc[RT2][4];
      const float* xa = w.A + ts * actH + (size_t)bt * H * 32;
      const float* xb = w.H0 + tp * actH + (size_t)bt * H * 32;
      skinny_gemm<RT2, true>(acc, P2, xa, xb, H / 16, wstage);
      reduce_store<RT2>(acc, red);
      __syncthreads();
      for (int idx = tid; idx < U * 32; idx += 256) {
        const int u = idx >> 5, b = idx & 31, j = c * U + u;
        float gir = red_sum<6 * U>(red, 0 * U + u, b) + gi0p[((bt * 3 + 0) * U + u) * 32 + b];
        float giz = red_sum<6 * U>(red, 1 * U + u, b) + gi0p[((bt * 3 + 1) * U + u) * 32 + b];
        float gin = red_sum<6 * U>(red, 2 * U + u, b) + gi0p[((bt * 3 + 2) * U + u) * 32 + b];
        float ghr = red_sum<6 * U>(red, 3 * U + u, b) + a.b_hh0[0 * H + j];
        float ghz = red_sum<6 * U>(red, 4 * U + u, b) + a.b_hh0[1 * H + j];
        float ghn = red_sum<6 * U>(red, 5 * U + u, b) + a.b_hh0[2 * H + j];
        float r = sigmoid_f(gir + ghr), z = sigmoid_f(giz + ghz);
        float n = tanhf(gin + r * ghn);
        float hp = ld_cg(xb + (size_t)j * 32 + b);
        float h = (1.f - z) * n + z * hp;
        w.H0[ts * actH + ((size_t)bt * H + j) * 32 + b] = h;
        if (w.save) {
          float* G = w.G0 + ((size_t)t * nbt + bt) * 4 * H * 32;
          G[(size_t)(0 * H + j) * 32 + b] = r; G[(size_t)(1 * H + j) * 32 + b] = z;
          G[(size_t)(2 * H + j) * 32 + b] = n; G[(size_t)(3 * H + j) * 32 + b] = ghn;
        }
      }
      __syncthreads();
    }
    if (!grid_sync(gb)) return;
    // ------------------------------------------------------------ stage 3 (GRU layer 1)
    for (int bt = 0; bt < nbt; ++bt) {
      float acc[RT2][4];
      const float* xa = w.H0 + ts * actH + (size_t)bt * H * 32;
      const float* xb = w.H1 + tp * actH + (size_t)bt * H * 32;
      skinny_gemm<RT2, true>(acc, P3, xa, xb, H / 16, wstage);
      reduce_store<RT2>(acc, red);
      __syncthreads();
      for (int idx = tid; idx < U * 32; idx += 256) {
        const int u = idx >> 5, b = idx & 31, j = c * U + u;
        float gir = red_sum<6 * U>(red, 0 * U + u, b) + a.b_ih1[0 * H + j];
        float giz = red_sum<6 * U>(red, 1 * U + u, b) + a.b_ih1[1 * H + j];
        float gin = red_sum<6 * U>(red, 2 * U + u, b) + a.b_ih1[2 * H + j];
        float ghr = red_sum<6 * U>(red, 3 * U + u, b) + a.b_hh1[0 * H + j];
        float ghz = red_sum<6 * U>(red, 4 * U + u, b) + a.b_hh1[1 * H + j];
        float ghn = red_sum<6 * U>(red, 5 * U + u, b) + a.b_hh1[2 * H + j];
        float r = sigmoid_f(gir + ghr), z = sigmoid_f(giz + ghz);
        float n = tanhf(gin + r * ghn);
        float hp = ld_cg(xb + (size_t)j * 32 + b);
        float h = (1.f - z) * n + z * hp;
        w.H1[ts * actH + ((size_t)bt * H + j) * 32 + b] = h;
        if (w.save) {
          float* G = w.G1 + ((size_t)t * nbt + bt) * 4 * H * 32;
          G[(size_t)(0 * H + j) * 32 + b] = r; G[(size_t)(1 * H + j) * 32 + b] = z;
          G[(size_t)(2 * H + j) * 32 + b] = n; G[(size_t)(3 * H + j) * 32 + b] = ghn;
        }
      }
      __syncthreads();
    }
    if (!grid_sync(gb)) return;
    // ------------------------------------------------------------ stage 4 (layer2 + pose integration)
    for (int bt = 0; bt < nbt; ++bt) {
      const float* x = w.H1 + ts * actH + (size_t)bt * H * 32;
      float* xpn = w.XP + tn * actX + (size_t)bt * K1P * 32;
      for (int tile = 0; tile < g.n4t; ++tile) {
        float acc[4][4];
        skinny_gemm<4, false>(acc, P4 + (size_t)tile * H * 16, x, x, H / 16, wstage);
        reduce_store<4>(acc, red);
        __syncthreads();
        for (int idx = tid; idx < 16 * 32; idx += 256) {
          const int r = idx >> 5, b = idx & 31;
          const int lr = tile * 16 + r, n = c * g.rpc + lr;
          if (lr < g.rpc && n < P_OUT) {
            float y = red_sum<16>(red, r, b) + a.b2[n];
            float p = y * a.out_std[n] + a.out_mean[n];        // modules.py:728
            const int bgl = bt * 32 + b;
            if (bgl < a.B) a.Y[((size_t)bgl * T + t) * P_OUT + n] = p;
            if (t + 1 < T) xpn[(size_t)n * 32 + b] = (p - a.in_mean[n]) / a.in_std[n];   // modules.py:713
            if (n < 6) rootv[n * 32 + b] = p;
          }
        }
        __syncthreads();
      }
      if (c == 0 && tid < 32) {
        const int b = tid, bgl = bt * 32 + b;
        if (bgl < a.B) {
          const float* rp = a.root_pos + ((size_t)bgl * T + (t - 1)) * 3;
          const float* rq = a.root_rot + ((size_t)bgl * T + (t - 1)) * 4;
          V3 pos = v3(rp[0], rp[1], rp[2]);
          Q4 q; q.w = rq[0]; q.x = rq[1]; q.y = rq[2]; q.z = rq[3];
          V3 vel = v3(rootv[0 * 32 + b], rootv[1 * 32 + b], rootv[2 * 32 + b]);
          V3 vrt = v3(rootv[3 * 32 + b], rootv[4 * 32 + b], rootv[5 * 32 + b]);
          V3 npos = quat_mul_vec(q, a.dt * vel) + pos;                               // modules.py:739
          Q4 nq = quat_mul(quat_from_helical(quat_mul_vec(q, a.dt * vrt)), q);      // modules.py:740
          float* op = a.root_pos + ((size_t)bgl * T + t) * 3;
          float* oq = a.root_rot + ((size_t)bgl * T + t) * 4;
          op[0] = npos.x; op[1] = npos.y; op[2] = npos.z;
          oq[0] = nq.w; oq[1] = nq.x; oq[2] = nq.y; oq[3] = nq.z;
          if (t + 1 < T) {
            const float* gp = a.gaze_pos + ((size_t)bgl * T + (t + 1)) * 3;
            V3 gd = quat_mul_vec(quat_inv(nq), v3(gp[0], gp[1], gp[2]) - npos);     // modules.py:696
            xpn[(size_t)(P_OUT + 0) * 32 + b] = (gd.x - a.in_mean[P_OUT + 0]) / a.in_std[P_OUT + 0];
            xpn[(size_t)(P_OUT + 1) * 32 + b] = (gd.y - a.in_mean[P_OUT + 1]) / a.in_std[P_OUT + 1];
            xpn[(size_t)(P_OUT + 2) * 32 + b] = (gd.z - a.in_mean[P_OUT + 2]) / a.in_std[P_OUT + 2];
          }
        }
      }
      __syncthreads();
    }
    if (t + 1 < T) { if (!grid_sync(gb)) return; }
  }
}

// ------------------------------------------------------------------ host side
static int check_fwd_args(const zeggs_decoder_fwd_args* a) {
  ZCHECK_ARG(a != nullptr, "decoder: null args");
  ZCHECK_ARG(a->B >= 1 && a->T >= 1, "decoder: bad B=%d T=%d", a->B, a->T);
  ZCHECK_ARG(a->H % 16 == 0 && pick_U(a->H) > 0, "decoder: hidden size %d unsupported (need H%%16==0, H<=1184)", a->H);
  ZCHECK_ARG(a->S >= 1 && a->Z >= 1 && a->S + a->Z <= 256, "decoder: bad S=%d Z=%d", a->S, a->Z);
  return ZEGGS_OK;
}

extern "C" size_t zeggs_decoder_packed_bytes(int H, int S, int Z) {
  if (H % 16 != 0 || pick_U(H) <= 0) return 0;
  DecGeom g = make_geom(1, H, S, Z);
  return g.packed_floats() * sizeof(float);
}

extern "C" int zeggs_decoder_pack_weights(const zeggs_decoder_fwd_args* a, float* packed, void* stream_) {
  CtxScope ctx_scope(a ? a->ctx : nullptr);
  int rc = check_fwd_args(a); if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  DecGeom g = make_geom(a->B, a->H, a->S, a->Z);
  pack_decoder_kernel<<<592, 256, 0, stream>>>(g, a->W0, a->W_ih0, a->W_hh0, a->W_ih1, a->W_hh1, a->W2, packed);
  count_launch();
  ZCHECK_LAUNCH();
  return ZEGGS_OK;
}

extern "C" size_t zeggs_decoder_workspace_bytes(int B, int T, int H, int S, int Z, int save) {
  if (H % 16 != 0 || pick_U(H) <= 0 || B < 1 || T < 1) return 0;
  DecGeom g = make_geom(B, H, S, Z);
  return make_ws(nullptr, g, T, save).bytes;
}

template <int U>
static int launch_fwd(const zeggs_decoder_fwd_args& a, const DecGeom& g, const DecWs& w, cudaStream_t stream) {
  constexpr int RT2 = (6 * U) / 4;
  size_t smem = (size_t)(8 * 2 * SkinnyCfg<RT2>::STG + 8 * 6 * U * 32 + g.nbt * 3 * U * 32 + 6 * 32) * sizeof(float);
  ZCHECK_CUDA(cudaFuncSetAttribute(decoder_fwd_kernel<U>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, nsm = 0, occ = 0;
  ZCHECK_CUDA(cudaGetDevice(&dev));
  ZCHECK_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
  ZCHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, decoder_fwd_kernel<U>, 256, smem));
  ZCHECK_ARG(occ * nsm >= g.G, "decoder: cooperative grid of %d CTAs does not fit (%d SMs x %d)", g.G, nsm, occ);
  void* args[] = {(void*)&a, (void*)&g, (void*)&w};
  ZCHECK_CUDA(cudaLaunchCooperativeKernel((void*)decoder_fwd_kernel<U>, dim3(g.G), dim3(256), args, smem, stream));
  count_launch();
  return ZEGGS_OK;
}

// s == NULL: the window starts from the CellStateEncoder and no state is exported (zeggs_decoder_window_fwd)
static int window_fwd(const zeggs_decoder_fwd_args* ap, const zeggs_decoder_state_args* s, void* stream_) {
  int rc = check_fwd_args(ap); if (rc) return rc;
  const zeggs_decoder_fwd_args& a = *ap;
  const float* h_init = s ? s->h_init : nullptr;
  const int* from_state = s ? s->init_from_state : nullptr;
  float* h_final = s ? s->h_final : nullptr;
  CtxScope ctx_scope(a.ctx);
  cudaStream_t stream = (cudaStream_t)stream_;
  DecGeom g = make_geom(a.B, a.H, a.S, a.Z);
  DecWs w = make_ws(a.workspace, g, a.T, a.save_for_backward);
  ZCHECK_ARG(a.workspace != nullptr && a.workspace_bytes >= w.bytes, "decoder: workspace too small (%zu < %zu)", a.workspace_bytes, w.bytes);
  ZCHECK_ARG(a.engine == 1 || a.packed != nullptr, "decoder: packed weights missing (call zeggs_decoder_pack_weights)");
  // zero: barrier words, the x_pose slots (k padding rows / batch padding columns) and the h slot 0
  ZCHECK_CUDA(cudaMemsetAsync(w.bar, 0, 256, stream));
  ZCHECK_CUDA(cudaMemsetAsync(w.XP, 0, (size_t)w.TS * g.nbt * K1P * 32 * sizeof(float), stream));
  ZCHECK_CUDA(cudaMemsetAsync(w.H0, 0, (size_t)g.nbt * a.H * 32 * sizeof(float), stream));
  ZCHECK_CUDA(cudaMemsetAsync(w.H1, 0, (size_t)g.nbt * a.H * 32 * sizeof(float), stream));
  const int slot1 = w.save ? 1 : 1;
  decoder_prologue_kernel<<<a.B, 256, 0, stream>>>(a, g, w.cse_in, w.XP + (size_t)slot1 * g.nbt * K1P * 32);
  count_launch();
  ZCHECK_LAUNCH();
  // CellStateEncoder (modules.py:238-243), unless every sample starts from the caller's state
  if (h_init == nullptr || from_state != nullptr) {
    rc = gemm_f32_auto(0, a.B, a.H, P_IN + a.Z, w.cse_in, P_IN + a.Z, a.Wc0, P_IN + a.Z, a.bc0, w.cse_h1, a.H, 1, 0, stream); if (rc) return rc;
    rc = gemm_f32_auto(0, a.B, a.H, a.H, w.cse_h1, a.H, a.Wc1, a.H, a.bc1, w.cse_h2, a.H, 1, 0, stream); if (rc) return rc;
    rc = gemm_f32_auto(0, a.B, 2 * a.H, a.H, w.cse_h2, a.H, a.Wc2, a.H, a.bc2, w.cse_out, 2 * a.H, 0, 0, stream); if (rc) return rc;
  }
  cse_scatter_kernel<<<ceil_div(a.B * 2 * a.H, 256), 256, 0, stream>>>(a.B, a.H, w.cse_out, h_init, from_state, w.H0, w.H1);
  count_launch();
  ZCHECK_LAUNCH();
  if (a.T > 1) {
    const int C = a.S + a.Z;
    size_t sm = (size_t)(C * 33 + 64 * (C + 1)) * sizeof(float);
    if (a.engine == 1) {
      // hoisted speech/style terms as two GEMMs (tcgen05 when a scratch buffer is set): S01[(t,b)][4H] =
      // cond_rows [(t,b)][C] . [W0[:, 1134:] ; W_ih0[:, H+1134:]]^T + [b0 ; b_ih0]
      ZCHECK_ARG(g.nbt == 1, "decoder tc engine handles one 32-sample batch tile (B <= 32); got B=%d", a.B);
      cond_rows_kernel<<<592, 256, 0, stream>>>(a, w.CONDR);
      count_launch();
      ZCHECK_LAUNCH();
      rc = decoder_fwd_tc_hoist(a, g, w, stream); if (rc) return rc;
      rc = decoder_fwd_tc_run(a, g, w, stream);
    } else {
      ZCHECK_CUDA(cudaFuncSetAttribute(cond_precompute_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      cond_precompute_kernel<<<dim3(a.T, g.nbt, ceil_div(4 * a.H, 64)), 256, sm, stream>>>(a, g, w.S01);
      count_launch();
      ZCHECK_LAUNCH();
      ScopedTimer tm("decoder_fwd", stream);
      if (g.U == 4) rc = launch_fwd<4>(a, g, w, stream); else rc = launch_fwd<8>(a, g, w, stream);
    }
    if (rc) return rc;
  }
  if (h_final) {
    // both engines leave frame t's state in slot (save ? t : t & 1) of H0 / H1; state carry runs without save, and with T == 1
    // slot 0 still holds the initial state
    const size_t slot = (size_t)((a.T - 1) & 1) * g.nbt * a.H * 32;
    state_gather_kernel<<<ceil_div(2 * a.B * a.H, 256), 256, 0, stream>>>(a.B, a.H, w.H0 + slot, w.H1 + slot, h_final);
    count_launch();
    ZCHECK_LAUNCH();
  }
  return ZEGGS_OK;
}

extern "C" int zeggs_decoder_window_fwd(const zeggs_decoder_fwd_args* a, void* stream) { return window_fwd(a, nullptr, stream); }

extern "C" int zeggs_decoder_window_fwd_state(const zeggs_decoder_fwd_args* a, const zeggs_decoder_state_args* s, void* stream) {
  ZCHECK_ARG(a != nullptr, "decoder: null args");
  ZCHECK_ARG(a->save_for_backward == 0, "decoder state carry is inference only: save_for_backward must be 0");
  ZCHECK_ARG(s == nullptr || s->init_from_state == nullptr || s->h_init != nullptr, "decoder: init_from_state given without h_init");
  return window_fwd(a, s, stream);
}

}  // namespace zeggs
