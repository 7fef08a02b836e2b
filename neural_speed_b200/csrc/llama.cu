// llama.cu -- device-resident decode/prefill step around the weight-only matmuls (SURVEY §8 f.1).
//
// Mirrors the Llama-family eval graph of the reference, models/llama/llama.cpp:190-720 (model_eval_internal):
//   inpL = get_rows(tok_embeddings, tokens)                                    :190
//   per layer: cur = rms_norm(inpL) * attn_norm                                :205-210
//              Q,K,V = mul_qkv / mul_mat                                       :212-240
//              rope(Q), rope(K) at position n_past + t (mode 0, pairs (2i,2i+1)) :351-355, ne_layers.c:9380-9396
//              K,V -> fp16 KV cache; attention = softmax(K Q / sqrt(hd)) V      :362-420 / :286-302 (ggml path)
//              inpFF = wo * attn + inpSA                                       :585-598
//              cur = rms_norm(inpFF) * ffn_norm ; cur = ffn_silu(cur) + inpFF  :601-698
//   logits = output * (rms_norm(inpL) * out_norm)                              :707-719
// Greedy sampling = argmax with the lowest index on ties (model_utils.cpp:2963-2985).
//
// One token (n_tokens == 1) is ONE CUDA graph: the token id and n_past live in device memory (`state`), so the same graph
// replays for every position; ns_llama_generate chains graph launches with the argmax feeding the next embedding
// lookup on the device -- no host round trip per token.
//
// Element-wise numerics follow the reference's ggml path: fp16 KV cache, Q and the softmax probabilities rounded to fp16
// before the K.Q and V.P dot products (ne_compute_forward_mul_mat_f16_f32), exp taken on the fp16-rounded argument and
// rounded to fp16 (table_exp_f16, ne_layers.c:8933-8937); rms_norm as kernel_ref.h:2199-2225.
#include <cuda_fp16.h>

#include <vector>

#include "nsb.cuh"

namespace {

struct Layer {
  const float* attn_norm = nullptr;
  const float* ffn_norm = nullptr;
  const ns_weight *wq = nullptr, *wk = nullptr, *wv = nullptr, *wo = nullptr, *w1 = nullptr, *w2 = nullptr, *w3 = nullptr;
};

constexpr int kAttnThreads = 128;

// x[t][:] = table[token[t]][:]
__global__ void __launch_bounds__(256) embed_kernel(const float* __restrict__ table, const int* __restrict__ tokens, int n_embd,
                                                    int n_vocab, float* __restrict__ x) {
  pdl_launch_dependents();
  pdl_wait();
  const int t = blockIdx.y;
  int tok = tokens[t];
  tok = tok < 0 ? 0 : (tok >= n_vocab ? n_vocab - 1 : tok);
  const float4* src = (const float4*)(table + (size_t)tok * n_embd);
  float4* dst = (float4*)(x + (size_t)t * n_embd);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_embd / 4; i += gridDim.x * blockDim.x) dst[i] = src[i];
}

// y = x / sqrt(mean(x^2) + eps) * w      (ne_rms_norm + ne_mul; kernel_ref.h:2199-2225 "simplified")
// One CTA per row; every thread issues ALL its loads (x and w, float4) before the first use, so the row costs one memory
// latency instead of one per loop trip (a single CTA is latency-bound, not bandwidth-bound).
template <int V4>  // float4 per thread: n <= 256 * 4 * V4
__global__ void __launch_bounds__(256) rmsnorm_kernel(const float* __restrict__ x, const float* __restrict__ w, float* __restrict__ y,
                                                      int n, float eps) {
  pdl_launch_dependents();
  const int n4 = n >> 2;
  float4 wv[V4];
#pragma unroll
  for (int j = 0; j < V4; ++j) {  // the norm weights do not depend on the previous kernel: fetch them before the wait
    const int i = threadIdx.x + j * 256;
    wv[j] = i < n4 ? ((const float4*)w)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  pdl_wait();
  const float4* xr = (const float4*)(x + (size_t)blockIdx.x * n);
  float4* yr = (float4*)(y + (size_t)blockIdx.x * n);
  float4 xv[V4];
#pragma unroll
  for (int j = 0; j < V4; ++j) {
    const int i = threadIdx.x + j * 256;
    xv[j] = i < n4 ? xr[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < V4; ++j) {
    ss = fmaf(xv[j].x, xv[j].x, ss);
    ss = fmaf(xv[j].y, xv[j].y, ss);
    ss = fmaf(xv[j].z, xv[j].z, ss);
    ss = fmaf(xv[j].w, xv[j].w, ss);
  }
  __shared__ float red[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) tot += red[i];
  const float inv = 1.f / sqrtf(tot / (float)n + eps);
#pragma unroll
  for (int j = 0; j < V4; ++j) {
    const int i = threadIdx.x + j * 256;
    if (i < n4) yr[i] = make_float4(xv[j].x * inv * wv[j].x, xv[j].y * inv * wv[j].y, xv[j].z * inv * wv[j].z, xv[j].w * inv * wv[j].w);
  }
}

// rope (mode 0) on q and k of every new token + append k,v to the fp16 cache.
// grid (n_head + n_head_kv, n_tokens), hd/2 threads.  pos = state[1] + t.
__global__ void rope_kv_kernel(float* __restrict__ q, int ldq, const float* __restrict__ k, int ldk, const float* __restrict__ v, int ldv,
                               __half* __restrict__ kc, __half* __restrict__ vc, const int* __restrict__ state, int n_head, int n_head_kv,
                               int hd, int n_ctx, float theta_scale, float freq_scale) {
  pdl_launch_dependents();
  pdl_wait();
  const int h = blockIdx.x, t = blockIdx.y, i = threadIdx.x;  // pair index
  const int pos = state[1] + t;
  // theta_base = p; repeated `theta_base *= theta_scale` (ne_layers.c:9321,9385): keep the same sequence of roundings
  float theta = (float)pos;
  for (int j = 0; j < i; ++j) theta *= theta_scale;
  theta *= freq_scale;
  float sn, cs;
  sincosf(theta, &sn, &cs);
  if (h < n_head) {
    float* p = q + (size_t)t * ldq + (size_t)h * hd + 2 * i;
    const float x0 = p[0], x1 = p[1];
    p[0] = x0 * cs - x1 * sn;
    p[1] = x0 * sn + x1 * cs;
  } else {
    const int hk = h - n_head;
    const float* p = k + (size_t)t * ldk + (size_t)hk * hd + 2 * i;
    const float x0 = p[0], x1 = p[1];
    if (pos < n_ctx) {
      __half* kd = kc + ((size_t)hk * n_ctx + pos) * hd + 2 * i;
      kd[0] = __float2half_rn(x0 * cs - x1 * sn);
      kd[1] = __float2half_rn(x0 * sn + x1 * cs);
      const float* pv = v + (size_t)t * ldv + (size_t)hk * hd + 2 * i;
      __half* vd = vc + ((size_t)hk * n_ctx + pos) * hd + 2 * i;
      vd[0] = __float2half_rn(pv[0]);
      vd[1] = __float2half_rn(pv[1]);
    }
  }
}

// one CTA per (head, new token): two-pass softmax over positions 0 .. state[1] + t, scores in shared memory.
// out[t][h*hd + d] = sum_i fp16(p_i) * V[i][d]
__global__ void __launch_bounds__(kAttnThreads) attn_kernel(const float* __restrict__ q, int ldq, const __half* __restrict__ kc,
                                                            const __half* __restrict__ vc, const int* __restrict__ state, float* __restrict__ out,
                                                            int ldo, int n_head, int n_head_kv, int hd, int n_ctx, float scale) {
  extern __shared__ float sm[];  // [hd] q (fp16-rounded) | [n_ctx] scores
  pdl_launch_dependents();
  pdl_wait();
  const int h = blockIdx.x, t = blockIdx.y;
  const int hk = h / (n_head / n_head_kv);
  int len = state[1] + t + 1;
  len = len > n_ctx ? n_ctx : len;
  float* sq = sm;
  float* sc = sm + hd;
  const float* qr = q + (size_t)t * ldq + (size_t)h * hd;
  for (int d = threadIdx.x; d < hd; d += blockDim.x) sq[d] = __half2float(__float2half_rn(qr[d]));
  __syncthreads();
  const __half* kh = kc + (size_t)hk * n_ctx * hd;
  const __half* vh = vc + (size_t)hk * n_ctx * hd;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  // pass 1: scores (one warp per position)
  float lmax = -INFINITY;
  for (int i = warp; i < len; i += nw) {
    const __half2* kr = (const __half2*)(kh + (size_t)i * hd);
    float acc = 0.f;
    for (int d2 = lane; d2 < hd / 2; d2 += 32) {
      const float2 kv = __half22float2(kr[d2]);
      acc = fmaf(sq[2 * d2], kv.x, acc);
      acc = fmaf(sq[2 * d2 + 1], kv.y, acc);
    }
    acc = warp_sum(acc) * scale;
    if (lane == 0) sc[i] = acc;
    lmax = fmaxf(lmax, acc);
  }
  __shared__ float red[kAttnThreads / 32];
  __shared__ float bcast;
  if (lane == 0) red[warp] = lmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int i = 1; i < nw; ++i) m = fmaxf(m, red[i]);
    bcast = m;
  }
  __syncthreads();
  const float mx = bcast;
  // exp on the fp16-rounded argument, result rounded to fp16 (table_exp_f16), sum in fp32
  float lsum = 0.f;
  for (int i = threadIdx.x; i < len; i += blockDim.x) {
    const float a = __half2float(__float2half_rn(sc[i] - mx));
    const float e = __half2float(__float2half_rn(expf(a)));
    sc[i] = e;
    lsum += e;
  }
  lsum = warp_sum(lsum);
  __syncthreads();
  if (lane == 0) red[warp] = lsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < nw; ++i) s += red[i];
    bcast = 1.f / s;
  }
  __syncthreads();
  const float inv = bcast;
  // pass 2: thread d accumulates sum_i fp16(p_i) * V[i][d]
  for (int d = threadIdx.x; d < hd; d += blockDim.x) {
    float acc = 0.f;
    for (int i = 0; i < len; ++i) {
      const float p = __half2float(__float2half_rn(sc[i] * inv));
      acc = fmaf(p, __half2float(vh[(size_t)i * hd + d]), acc);
    }
    out[(size_t)t * ldo + (size_t)h * hd + d] = acc;
  }
}

// Decode-shaped attention for head sizes 64 / 128: kAW warps per (head, token); a warp streams whole K/V rows (one 4- or 8-byte
// load per lane), four rows in flight; with FUSE (single new token) the kernel also applies RoPE to its q head and to the
// new k row and appends k,v to the cache, so rope_kv_kernel is not launched.
constexpr int kAW = 16;  // warps per CTA: the kernel is a chain of dependent cache-row loads, more warps = more rows in flight
template <int HD, bool FUSE>
__global__ void __launch_bounds__(kAW * 32) attn_fast_kernel(const float* __restrict__ q, int ldq, const float* __restrict__ knew, int ldk,
                                                        const float* __restrict__ vnew, int ldv, __half* __restrict__ kc,
                                                        __half* __restrict__ vc, const int* __restrict__ state, float* __restrict__ out, int ldo,
                                                        int n_head, int n_head_kv, int n_ctx, float scale, float theta_scale,
                                                        float freq_scale) {
  constexpr int EPL = HD / 32;  // elements per lane
  extern __shared__ float sm[];  // [HD] q | [HD] new k | [HD] new v | [kAW][HD] partial out | [n_ctx] scores
  float* sq = sm;
  float* sk = sm + HD;
  float* sv = sm + 2 * HD;
  float* part = sm + 3 * HD;
  float* sc = sm + 3 * HD + kAW * HD;
  pdl_launch_dependents();
  pdl_wait();
  const int h = blockIdx.x, t = blockIdx.y;
  const int group = n_head / n_head_kv, hk = h / group;
  const int pos = state[1] + t;
  int len = pos + 1;
  len = len > n_ctx ? n_ctx : len;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __half* kh = kc + (size_t)hk * n_ctx * HD;
  __half* vh = vc + (size_t)hk * n_ctx * HD;
  const float* qr = q + (size_t)t * ldq + (size_t)h * HD;
  if (FUSE) {
    if (threadIdx.x < HD / 2) {
      const int i = threadIdx.x;
      float theta = (float)pos;
      for (int j = 0; j < i; ++j) theta *= theta_scale;  // ne_layers.c:9385: same sequence of roundings
      theta *= freq_scale;
      float sn, cs;
      sincosf(theta, &sn, &cs);
      const float q0 = qr[2 * i], q1 = qr[2 * i + 1];
      sq[2 * i] = __half2float(__float2half_rn(q0 * cs - q1 * sn));
      sq[2 * i + 1] = __half2float(__float2half_rn(q0 * sn + q1 * cs));
      const float* kr = knew + (size_t)t * ldk + (size_t)hk * HD;
      const float k0 = kr[2 * i], k1 = kr[2 * i + 1];
      const __half r0 = __float2half_rn(k0 * cs - k1 * sn), r1 = __float2half_rn(k0 * sn + k1 * cs);
      sk[2 * i] = __half2float(r0);
      sk[2 * i + 1] = __half2float(r1);
      const float* vr = vnew + (size_t)t * ldv + (size_t)hk * HD;
      const __half w0 = __float2half_rn(vr[2 * i]), w1 = __float2half_rn(vr[2 * i + 1]);
      sv[2 * i] = __half2float(w0);
      sv[2 * i + 1] = __half2float(w1);
      if (h % group == 0 && pos < n_ctx) {  // one CTA per kv head appends to the cache
        *(__half2*)(kh + (size_t)pos * HD + 2 * i) = __halves2half2(r0, r1);
        *(__half2*)(vh + (size_t)pos * HD + 2 * i) = __halves2half2(w0, w1);
      }
    }
  } else {
    for (int d = threadIdx.x; d < HD; d += blockDim.x) sq[d] = __half2float(__float2half_rn(qr[d]));
  }
  __syncthreads();
  float ql[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) ql[e] = sq[lane * EPL + e];
  const int ncache = FUSE ? len - 1 : len;  // rows read from the cache; the new row comes from shared memory when fused

  auto load_row = [&](const __half* base, int i, float* dst) {
    if (EPL == 4) {
      const uint2 u = *(const uint2*)(base + (size_t)i * HD + lane * 4);
      const float2 a = __half22float2(*(const __half2*)&u.x), b = __half22float2(*(const __half2*)&u.y);
      dst[0] = a.x, dst[1] = a.y, dst[2] = b.x, dst[3] = b.y;
    } else {
      const __half2 u = *(const __half2*)(base + (size_t)i * HD + lane * 2);
      const float2 a = __half22float2(u);
      dst[0] = a.x, dst[1] = a.y;
    }
  };
  // pass 1: scores
  for (int i0 = warp * 4; i0 < ncache; i0 += kAW * 4) {
    float kr[4][EPL];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (i0 + u < ncache) load_row(kh, i0 + u, kr[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (i0 + u < ncache) {  // warp-uniform
        float acc = 0.f;
#pragma unroll
        for (int e = 0; e < EPL; ++e) acc = fmaf(ql[e], kr[u][e], acc);
        acc = warp_sum(acc);
        if (lane == 0) sc[i0 + u] = acc * scale;
      }
    }
  }
  if (FUSE && warp == 0 && len - 1 == ncache) {
    float acc = 0.f;
#pragma unroll
    for (int e = 0; e < EPL; ++e) acc = fmaf(ql[e], sk[lane * EPL + e], acc);
    acc = warp_sum(acc);
    if (lane == 0) sc[len - 1] = acc * scale;
  }
  __syncthreads();
  __shared__ float red[kAW];
  __shared__ float bcast;
  float lmax = -INFINITY;
  for (int i = threadIdx.x; i < len; i += blockDim.x) lmax = fmaxf(lmax, sc[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
  if (lane == 0) red[warp] = lmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int i = 1; i < kAW; ++i) m = fmaxf(m, red[i]);
    bcast = m;
  }
  __syncthreads();
  const float mx = bcast;
  float lsum = 0.f;
  for (int i = threadIdx.x; i < len; i += blockDim.x) {
    const float a = __half2float(__float2half_rn(sc[i] - mx));
    const float e = __half2float(__float2half_rn(expf(a)));  // table_exp_f16 (ne_layers.c:8933-8937)
    sc[i] = e;
    lsum += e;
  }
  lsum = warp_sum(lsum);
  __syncthreads();
  if (lane == 0) red[warp] = lsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s2 = 0.f;
    for (int i = 0; i < kAW; ++i) s2 += red[i];
    bcast = 1.f / s2;
  }
  __syncthreads();
  const float inv = bcast;
  // pass 2: each warp accumulates its rows, lanes own EPL output elements; then the 8 partials are summed
  float acc[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) acc[e] = 0.f;
  for (int i0 = warp * 4; i0 < ncache; i0 += kAW * 4) {
    float vr[4][EPL];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (i0 + u < ncache) load_row(vh, i0 + u, vr[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (i0 + u < ncache) {
        const float p = __half2float(__float2half_rn(sc[i0 + u] * inv));
#pragma unroll
        for (int e = 0; e < EPL; ++e) acc[e] = fmaf(p, vr[u][e], acc[e]);
      }
  }
  if (FUSE && warp == 0 && len - 1 == ncache) {
    const float p = __half2float(__float2half_rn(sc[len - 1] * inv));
#pragma unroll
    for (int e = 0; e < EPL; ++e) acc[e] = fmaf(p, sv[lane * EPL + e], acc[e]);
  }
#pragma unroll
  for (int e = 0; e < EPL; ++e) part[warp * HD + lane * EPL + e] = acc[e];
  __syncthreads();
  for (int d = threadIdx.x; d < HD; d += blockDim.x) {
    float s2 = 0.f;
#pragma unroll
    for (int w = 0; w < kAW; ++w) s2 += part[w * HD + d];
    out[(size_t)t * ldo + (size_t)h * HD + d] = s2;
  }
}

// ---- decode attention: K / V of the head staged by TMA, split over the context ---------------------------------------------------
// One new token (llama.cpp:286-302 with N = 1; RoPE of q and of the new k row and the KV append fused in, as attn_fast_kernel<FUSE>).
// grid (n_head, ceil(n_ctx / 256)); CTA (h, s) owns cached positions [256 s, 256 s + 256) of head h and returns at once when the
// sequence has not reached its range (the position lives in device memory: one CUDA graph serves every position).  The rows of a
// head are contiguous in the cache ([kv head][n_ctx][hd] fp16), so the CTA's whole K and V ranges arrive as TWO cp.async.bulk copies
// (<= 64 KB each) on one mbarrier: a single global-memory latency per launch instead of a chain of dependent row loads -- the old
// kernel spent 2-3 round trips per pass at 100-200 positions.  Scores, soft_max and P.V then run out of shared memory.
// One active range (<= 256 positions): exactly the reference arithmetic (global maximum, e = fp16(exp(fp16(s - max))),
// p = fp16(e / sum), fp32 sums).  Several: every CTA leaves {max, sum e, sum e V} of its range, the last one to arrive (ticket per
// head) merges them with exp(max_s - max) weights -- same values up to the fp16 rounding of p (5e-4 relative).
// Bound: latency at short contexts; HBM (2 x len x hd x 2 B per kv head) at long ones, spread over n_head x ceil(len / 256) CTAs.
constexpr int kSplitKeys = 256;
constexpr int kDW = 16;  // warps per CTA
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
template <int HD>
static constexpr size_t attn_decode_smem() {
  return (size_t)2 * kSplitKeys * HD * 2 + (size_t)(3 + kDW) * HD * 4 + (size_t)(kSplitKeys + 8) * 4 + 16;
}
template <int HD>
__global__ void __launch_bounds__(kDW * 32) attn_decode_kernel(const float* __restrict__ q, const float* __restrict__ knew,
                                                            const float* __restrict__ vnew, __half* __restrict__ kc, __half* __restrict__ vc,
                                                            const int* __restrict__ state, float* __restrict__ out, float* __restrict__ part_ws,
                                                            unsigned* __restrict__ tickets, int n_head, int n_head_kv, int n_ctx, int nsplit,
                                                            float scale, float theta_scale, float freq_scale) {
  constexpr int EPL = HD / 32;
  extern __shared__ __align__(128) unsigned char smraw[];
  __half* Kt = reinterpret_cast<__half*>(smraw);  // [kSplitKeys][HD]
  __half* Vt = Kt + kSplitKeys * HD;
  float* sq = reinterpret_cast<float*>(Vt + kSplitKeys * HD);
  float* sk = sq + HD;
  float* sv = sk + HD;
  float* part = sv + HD;         // [kDW][HD]
  float* sc = part + kDW * HD;   // [kSplitKeys + 1]: scores of the range (+ the new row)
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(sc + kSplitKeys + 8);
  __shared__ float red[kDW];
  __shared__ float bcast;
  __shared__ int last_flag;
  pdl_launch_dependents();
  // The position was written by the PREVIOUS token's argmax kernel (an earlier graph launch / an H2D copy ahead of this eval's
  // first kernel), never by a kernel of this token: it may be read before griddepcontrol.wait.  CTAs whose range the sequence
  // has not reached leave at once, without holding 141 KB of an SM until the Q/K/V launch in front of this one has drained.
  const int h = blockIdx.x, split = blockIdx.y;
  const int group = n_head / n_head_kv, hk = h / group;
  const int pos = state[1];
  const int len = min(pos + 1, n_ctx);
  const int nact = (len + kSplitKeys - 1) / kSplitKeys;
  if (split >= nact) return;
  const int i0 = split * kSplitKeys, i1 = min(len, i0 + kSplitKeys);
  const bool has_new = (i1 == len) && pos < n_ctx;  // the token being evaluated sits in this range: its k / v come from registers
  const int ncache = (has_new ? i1 - 1 : i1) - i0;  // rows read from the cache
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __half* kh = kc + (size_t)hk * n_ctx * HD;
  __half* vh = vc + (size_t)hk * n_ctx * HD;
  const uint32_t bar_a = smem_addr(bar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_a), "r"(1) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // the cached rows of this range were written by earlier tokens' launches: their copies start before the wait as well and
    // overlap the tail of the Q/K/V launch
    if (ncache > 0) {
      const uint32_t bytes = (uint32_t)ncache * HD * 2;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(2 * bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(Kt)),
                   "l"(kh + (size_t)i0 * HD), "r"(bytes), "r"(bar_a)
                   : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(Vt)),
                   "l"(vh + (size_t)i0 * HD), "r"(bytes), "r"(bar_a)
                   : "memory");
    }
  }
  __syncthreads();
  pdl_wait();  // q, k, v of the new token come from the launch in front
  // RoPE of this head's q (every range needs it) and of the new k row; KV append by one CTA per kv head -- while the copies fly
  if (threadIdx.x < HD / 2) {
    const int i = threadIdx.x;
    float theta = (float)pos;
    for (int j = 0; j < i; ++j) theta *= theta_scale;  // ne_layers.c:9385: same sequence of roundings
    theta *= freq_scale;
    float sn, cs;
    sincosf(theta, &sn, &cs);
    const float* qr = q + (size_t)h * HD;
    const float q0 = qr[2 * i], q1 = qr[2 * i + 1];
    sq[2 * i] = __half2float(__float2half_rn(q0 * cs - q1 * sn));
    sq[2 * i + 1] = __half2float(__float2half_rn(q0 * sn + q1 * cs));
    if (has_new) {
      const float* kr = knew + (size_t)hk * HD;
      const float k0 = kr[2 * i], k1 = kr[2 * i + 1];
      const __half r0 = __float2half_rn(k0 * cs - k1 * sn), r1 = __float2half_rn(k0 * sn + k1 * cs);
      sk[2 * i] = __half2float(r0);
      sk[2 * i + 1] = __half2float(r1);
      const float* vr = vnew + (size_t)hk * HD;
      const __half w0 = __float2half_rn(vr[2 * i]), w1 = __float2half_rn(vr[2 * i + 1]);
      sv[2 * i] = __half2float(w0);
      sv[2 * i + 1] = __half2float(w1);
      if (h % group == 0) {
        *reinterpret_cast<__half2*>(kh + (size_t)pos * HD + 2 * i) = __halves2half2(r0, r1);
        *reinterpret_cast<__half2*>(vh + (size_t)pos * HD + 2 * i) = __halves2half2(w0, w1);
      }
    }
  }
  __syncthreads();
  float ql[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) ql[e] = sq[lane * EPL + e];
  if (ncache > 0) {
    uint32_t ok;
    do {
      asm volatile(
          "{\n"
          ".reg .pred p;\n"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
          "selp.u32 %0, 1, 0, p;\n"
          "}\n"
          : "=r"(ok)
          : "r"(bar_a), "r"(0)
          : "memory");
    } while (!ok);
  }
  auto row = [&](const __half* base, int r, float* dst) {
    if (EPL == 4) {
      const uint2 u = *reinterpret_cast<const uint2*>(base + (size_t)r * HD + lane * 4);
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      dst[0] = a.x, dst[1] = a.y, dst[2] = b.x, dst[3] = b.y;
    } else {
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(base + (size_t)r * HD + lane * 2));
      dst[0] = a.x, dst[1] = a.y;
    }
  };
  // pass 1: scores of the range
  for (int r = warp; r < ncache; r += kDW) {
    float kr[EPL];
    row(Kt, r, kr);
    float acc = 0.f;
#pragma unroll
    for (int e = 0; e < EPL; ++e) acc = fmaf(ql[e], kr[e], acc);
    acc = warp_sum(acc);
    if (lane == 0) sc[r] = acc * scale;
  }
  if (has_new && warp == kDW - 1) {
    float acc = 0.f;
#pragma unroll
    for (int e = 0; e < EPL; ++e) acc = fmaf(ql[e], sk[lane * EPL + e], acc);
    acc = warp_sum(acc);
    if (lane == 0) sc[ncache] = acc * scale;
  }
  __syncthreads();
  const int nloc = ncache + (has_new ? 1 : 0);
  float lmax = -INFINITY;
  for (int i = threadIdx.x; i < nloc; i += blockDim.x) lmax = fmaxf(lmax, sc[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
  if (lane == 0) red[warp] = lmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int i = 1; i < kDW; ++i) m = fmaxf(m, red[i]);
    bcast = m;
  }
  __syncthreads();
  const float mx = bcast;
  float lsum = 0.f;
  for (int i = threadIdx.x; i < nloc; i += blockDim.x) {
    const float a = __half2float(__float2half_rn(sc[i] - mx));
    const float e = __half2float(__float2half_rn(expf(a)));  // table_exp_f16 (ne_layers.c:8933-8937)
    sc[i] = e;
    lsum += e;
  }
  lsum = warp_sum(lsum);
  __syncthreads();
  if (lane == 0) red[warp] = lsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s2 = 0.f;
    for (int i = 0; i < kDW; ++i) s2 += red[i];
    bcast = s2;
  }
  __syncthreads();
  const float lrange = bcast;
  const bool single = nact == 1;
  const float inv = 1.f / lrange;
  // pass 2: sum p V over the range; warps own rows, lanes own EPL output elements
  float acc[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) acc[e] = 0.f;
  for (int r = warp; r < ncache; r += kDW) {
    float vr[EPL];
    row(Vt, r, vr);
    const float p = single ? __half2float(__float2half_rn(sc[r] * inv)) : sc[r];
#pragma unroll
    for (int e = 0; e < EPL; ++e) acc[e] = fmaf(p, vr[e], acc[e]);
  }
  if (has_new && warp == kDW - 1) {
    const float p = single ? __half2float(__float2half_rn(sc[ncache] * inv)) : sc[ncache];
#pragma unroll
    for (int e = 0; e < EPL; ++e) acc[e] = fmaf(p, sv[lane * EPL + e], acc[e]);
  }
#pragma unroll
  for (int e = 0; e < EPL; ++e) part[warp * HD + lane * EPL + e] = acc[e];
  __syncthreads();
  float mine = 0.f;
  if (threadIdx.x < HD) {
#pragma unroll
    for (int w = 0; w < kDW; ++w) mine += part[w * HD + threadIdx.x];
  }
  if (single) {
    if (threadIdx.x < HD) out[(size_t)h * HD + threadIdx.x] = mine;
    return;
  }
  // several ranges: leave {sum e V, max, sum e}; the last CTA of the head merges
  float* mypart = part_ws + ((size_t)h * nsplit + split) * (HD + 2);
  if (threadIdx.x < HD) mypart[threadIdx.x] = mine;
  if (threadIdx.x == 0) {
    mypart[HD] = mx;
    mypart[HD + 1] = lrange;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last_flag = (atomicAdd(&tickets[h], 1u) == (unsigned)(nact - 1)) ? 1 : 0;
  __syncthreads();
  if (!last_flag) return;
  __threadfence();
  if (threadIdx.x < HD) {
    const float* base = part_ws + (size_t)h * nsplit * (HD + 2);
    float gm = -INFINITY;
    for (int s2 = 0; s2 < nact; ++s2) gm = fmaxf(gm, __ldcg(base + (size_t)s2 * (HD + 2) + HD));
    float num = 0.f, den = 0.f;
    for (int s2 = 0; s2 < nact; ++s2) {
      const float w = expf(__ldcg(base + (size_t)s2 * (HD + 2) + HD) - gm);
      num = fmaf(w, __ldcg(base + (size_t)s2 * (HD + 2) + threadIdx.x), num);
      den = fmaf(w, __ldcg(base + (size_t)s2 * (HD + 2) + HD + 1), den);
    }
    out[(size_t)h * HD + threadIdx.x] = num / den;
  }
  if (threadIdx.x == 0) tickets[h] = 0u;  // ready for the next launch (graph replay)
}

// ---- prompt attention on the tensor cores ------------------------------------------------------------------------------------
// The ggml attention of the reference for N > 1 new tokens (llama.cpp:286-302: KQ = mul_mat(K, Q) -> scale -> diag_mask_inf ->
// soft_max -> mul_mat(V, KQ_soft_max); ne_compute_forward_mul_mat_f16_f32 rounds Q and the probabilities to fp16 and sums the
// fp16 x fp16 products in fp32, ne_layers.c:6943-7083; soft_max rounds (s - max) and exp() to fp16, :8887-8954) as a causal
// two-pass kernel on mma.sync.m16n8k16 f16 -> f32 (the same operand types and accumulator as the reference's dot products):
//   pass A  S = Q K^T tile by tile, row maxima (the reference's soft_max uses the GLOBAL row maximum, not a running one)
//   pass B  S again, e = fp16(exp(fp16(s - max))), l += e, O += e V (e is an exact fp16 value: the products are exact), out = O / l
// (difference to the reference: it rounds e / l to fp16 before the V product; here the division happens once, in fp32, after it).
// CTA = 64 query rows of one head (4 warps x 16 rows); K / V tiles of 64 keys staged in shared memory with 16-byte padded rows
// (conflict-free 32-bit B-fragment loads for K, ldmatrix.trans for V); every q-tile of a head re-reads that head's K / V through L2.
// Bound: tensor pipe / shared-memory bandwidth (K and V of one head are 0.5 MB at 2048 positions -- L2 resident).
constexpr int kAttnMmaRows = 64, kAttnMmaKeys = 64;
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void mma_f16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
template <int HD>
__global__ void __launch_bounds__(128) attn_mma_kernel(const float* __restrict__ q, int ldq, const __half* __restrict__ kc,
                                                       const __half* __restrict__ vc, const int* __restrict__ state, float* __restrict__ out,
                                                       int ldo, int n_head, int n_head_kv, int n_ctx, int m, float scale) {
  constexpr int LD = HD + 8;  // halves per shared-memory row: 16 bytes of padding rotate the banks by 4 words per row
  constexpr int KS = HD / 16, NT = HD / 8;
  __shared__ __align__(16) __half Ks[kAttnMmaKeys * LD];
  __shared__ __align__(16) __half Vs[kAttnMmaKeys * LD];
  pdl_launch_dependents();
  pdl_wait();
  const int h = blockIdx.y, hk = h / (n_head / n_head_kv);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
  const int pos0 = state[1];
  const int q0 = blockIdx.x * kAttnMmaRows;
  const int row0 = q0 + warp * 16 + g, row1 = row0 + 8;  // this thread's two query rows (token indices of the batch)
  const int total = min(pos0 + m, n_ctx);                // keys that exist
  const __half* kh = kc + (size_t)hk * n_ctx * HD;
  const __half* vh = vc + (size_t)hk * n_ctx * HD;

  // Q A-fragments, rounded to fp16 as the reference's mul_mat does with src1 (rows past the batch: zeros)
  uint32_t qa[KS][4];
  {
    const float* q0p = q + (size_t)row0 * ldq + (size_t)h * HD;
    const float* q1p = q + (size_t)row1 * ldq + (size_t)h * HD;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      const int c = ks * 16 + 2 * t4;
      const float2 a0 = row0 < m ? *reinterpret_cast<const float2*>(q0p + c) : make_float2(0.f, 0.f);
      const float2 a1 = row1 < m ? *reinterpret_cast<const float2*>(q1p + c) : make_float2(0.f, 0.f);
      const float2 a2 = row0 < m ? *reinterpret_cast<const float2*>(q0p + c + 8) : make_float2(0.f, 0.f);
      const float2 a3 = row1 < m ? *reinterpret_cast<const float2*>(q1p + c + 8) : make_float2(0.f, 0.f);
      qa[ks][0] = pack_h2(a0.x, a0.y);
      qa[ks][1] = pack_h2(a1.x, a1.y);
      qa[ks][2] = pack_h2(a2.x, a2.y);
      qa[ks][3] = pack_h2(a3.x, a3.y);
    }
  }
  const int last_row = min(q0 + kAttnMmaRows, m) - 1;
  const int nkt = min(pos0 + last_row, total - 1) / kAttnMmaKeys + 1;  // key tiles this CTA needs
  const int warp_last_key = pos0 + q0 + warp * 16 + 15;                // beyond it every key is masked for the whole warp

  auto load_tile = [&](const __half* base, __half* dst, int key0) {
    constexpr int C16 = HD / 8;  // 16-byte chunks per row
#pragma unroll
    for (int i = 0; i < kAttnMmaKeys * C16 / 128; ++i) {
      const int idx = i * 128 + (int)threadIdx.x;
      const int r = idx / C16, c = idx % C16;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (key0 + r < total) v = *reinterpret_cast<const uint4*>(base + (size_t)(key0 + r) * HD + c * 8);
      *reinterpret_cast<uint4*>(dst + r * LD + c * 8) = v;
    }
  };
  auto scores = [&](float (&s)[8][4]) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) s[j][c] = 0.f;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const __half* kr = Ks + (j * 8 + g) * LD + ks * 16 + 2 * t4;
        mma_f16_16816(s[j], qa[ks], *reinterpret_cast<const uint32_t*>(kr), *reinterpret_cast<const uint32_t*>(kr + 8));
      }
  };

  // ---- pass A: row maxima of the masked, scaled scores
  float mx0 = -INFINITY, mx1 = -INFINITY;
  for (int kt = 0; kt < nkt; ++kt) {
    __syncthreads();
    load_tile(kh, Ks, kt * kAttnMmaKeys);
    __syncthreads();
    if (kt * kAttnMmaKeys > warp_last_key) continue;
    float s[8][4];
    scores(s);
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int key = kt * kAttnMmaKeys + j * 8 + 2 * t4 + (c & 1);
        const int row = (c < 2) ? row0 : row1;
        if (key <= pos0 + row && key < total) {
          if (c < 2) mx0 = fmaxf(mx0, s[j][c] * scale);
          else mx1 = fmaxf(mx1, s[j][c] * scale);
        }
      }
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  if (row0 >= m) mx0 = 0.f;  // rows past the batch: nothing valid, nothing stored
  if (row1 >= m) mx1 = 0.f;

  // ---- pass B: e = fp16(exp(fp16(s - max))), l = sum e, O = sum e V
  float o[NT][4];
#pragma unroll
  for (int n = 0; n < NT; ++n)
#pragma unroll
    for (int c = 0; c < 4; ++c) o[n][c] = 0.f;
  float l0 = 0.f, l1 = 0.f;
  for (int kt = 0; kt < nkt; ++kt) {
    __syncthreads();
    load_tile(kh, Ks, kt * kAttnMmaKeys);
    load_tile(vh, Vs, kt * kAttnMmaKeys);
    __syncthreads();
    if (kt * kAttnMmaKeys > warp_last_key) continue;
    float s[8][4];
    scores(s);
    uint32_t pe[8][2];  // per 8-key tile: (row0: keys 2t4, 2t4+1), (row1: same keys) as fp16 pairs
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float e[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int key = kt * kAttnMmaKeys + j * 8 + 2 * t4 + (c & 1);
        const int row = (c < 2) ? row0 : row1;
        const bool valid = key <= pos0 + row && key < total && row < m;
        const float a = __half2float(__float2half_rn(s[j][c] * scale - (c < 2 ? mx0 : mx1)));
        e[c] = valid ? __half2float(__float2half_rn(expf(a))) : 0.f;  // table_exp_f16 (ne_layers.c:8933-8937)
      }
      l0 += e[0] + e[1];
      l1 += e[2] + e[3];
      pe[j][0] = pack_h2(e[0], e[1]);
      pe[j][1] = pack_h2(e[2], e[3]);
    }
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {  // 16 keys per step: P as the A operand straight from the score accumulators
      const uint32_t pa[4] = {pe[2 * kk][0], pe[2 * kk][1], pe[2 * kk + 1][0], pe[2 * kk + 1][1]};
      const __half* vrow = Vs + (kk * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * LD + 8 * (lane >> 4);
#pragma unroll
      for (int n2 = 0; n2 < NT / 2; ++n2) {
        uint32_t b0, b1, b2, b3;
        const uint32_t addr = (uint32_t)__cvta_generic_to_shared(vrow + n2 * 16);
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3) : "r"(addr));
        mma_f16_16816(o[2 * n2], pa, b0, b1);
        mma_f16_16816(o[2 * n2 + 1], pa, b2, b3);
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.f / l0, i1 = 1.f / l1;
#pragma unroll
  for (int n = 0; n < NT; ++n) {
    const int d = n * 8 + 2 * t4;
    if (row0 < m) *reinterpret_cast<float2*>(out + (size_t)row0 * ldo + (size_t)h * HD + d) = make_float2(o[n][0] * i0, o[n][1] * i0);
    if (row1 < m) *reinterpret_cast<float2*>(out + (size_t)row1 * ldo + (size_t)h * HD + d) = make_float2(o[n][2] * i1, o[n][3] * i1);
  }
}

// greedy pick: index of the maximum, lowest index on ties (model_utils.cpp:2963-2985); also advances the device-side
// position.  kArgmaxBlocks CTAs scan slices (all loads in flight at once); the last CTA to finish (ticket) merges the
// partial results.  state[3] = pick; when `advance`: state[0] = pick, state[1] += n_tokens, record[state[2]++] = pick.
constexpr int kArgmaxBlocks = 32;
__device__ __forceinline__ void argmax_merge(float& best, int& bi, float ov, int oi) {
  if (ov > best || (ov == best && oi < bi)) {
    best = ov;
    bi = oi;
  }
}
__global__ void __launch_bounds__(256) argmax_kernel(const float* __restrict__ logits, int n, int* __restrict__ state, int n_tokens,
                                                     int advance, int* __restrict__ record, float* __restrict__ pval, int* __restrict__ pidx,
                                                     unsigned* __restrict__ ticket) {
  pdl_launch_dependents();
  pdl_wait();
  const int per = (n + kArgmaxBlocks - 1) / kArgmaxBlocks;
  const int lo = blockIdx.x * per, hi = min(n, lo + per);
  float best = -INFINITY;
  int bi = 0x7fffffff;
  constexpr int U = 4;
  for (int i0 = lo + threadIdx.x; i0 < hi; i0 += 256 * U) {
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = (i0 + u * 256 < hi) ? logits[i0 + u * 256] : -INFINITY;
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (i0 + u * 256 < hi) argmax_merge(best, bi, v[u], i0 + u * 256);
  }
  __shared__ float sv[8];
  __shared__ int si[8];
  __shared__ bool last;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) argmax_merge(best, bi, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, bi, o));
  if ((threadIdx.x & 31) == 0) {
    sv[threadIdx.x >> 5] = best;
    si[threadIdx.x >> 5] = bi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) argmax_merge(best, bi, sv[w], si[w]);
    pval[blockIdx.x] = best;
    pidx[blockIdx.x] = bi;
    __threadfence();
    last = atomicAdd(ticket, 1u) == kArgmaxBlocks - 1;
  }
  __syncthreads();
  if (!last || threadIdx.x != 0) return;
  __threadfence();
  best = -INFINITY;
  bi = 0x7fffffff;
  for (int b2 = 0; b2 < kArgmaxBlocks; ++b2) argmax_merge(best, bi, ((volatile float*)pval)[b2], ((volatile int*)pidx)[b2]);
  if (bi == 0x7fffffff) bi = 0;  // all NaN / -inf: the reference's loop keeps index 0
  *ticket = 0u;                  // ready for the next launch
  state[3] = bi;
  if (advance) {
    state[0] = bi;
    state[1] += n_tokens;
    if (record) record[state[2]++] = bi;
  }
}

}  // namespace

struct ns_llama {
  ns_llama_hparams hp;
  cudaStream_t st;
  std::vector<Layer> layers;
  float* tok_embd = nullptr;
  float* out_norm = nullptr;
  const ns_weight* output = nullptr;
  std::vector<void*> owned;  // device allocations freed with the context
  __half *kc = nullptr, *vc = nullptr;
  int* state = nullptr;   // device: {token, n_past, n_recorded, last_pick}
  int* tokens = nullptr;  // device: prompt tokens of the current eval
  int* record = nullptr;  // device: generated tokens
  float* am_val = nullptr;  // argmax partials
  int* am_idx = nullptr;
  unsigned* am_ticket = nullptr;
  int m_cap = 0;
  size_t attn_attr = 0, fast_attr = 0;  // dynamic shared memory already granted to the attention kernels
  int dec_attr = 0;                     // attn_decode_kernel attribute set for this context's device
  float* attn_part = nullptr;           // split-context decode attention: [n_head][nsplit][hd + 2] partials
  unsigned* attn_tickets = nullptr;     // [n_head]
  int attn_nsplit = 0;
  int exact_prefill = 0;               // ns_llama_set_exact_prefill
  float *x = nullptr, *xn = nullptr, *qkv = nullptr, *attn = nullptr, *tmp = nullptr, *logits = nullptr;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  cudaGraphExec_t decode_exec = nullptr;
  cudaGraph_t decode_graph = nullptr;
  int tap_layer = -1;  // ns_llama_set_tap: copies of this layer's q|k|v (before RoPE) and attention output
  float *tap_qkv = nullptr, *tap_attn = nullptr;
  int tap_rows = 0;
  int* h_state = nullptr;  // pinned host staging
  float* h_logits = nullptr;
};

static void* dev_alloc(ns_llama* c, size_t bytes) {
  void* p = nullptr;
  if (cudaMalloc(&p, bytes) != cudaSuccess) {
    ns_set_error("ns_llama: cudaMalloc(%zu) failed", bytes);
    return nullptr;
  }
  c->owned.push_back(p);
  return p;
}

// release one allocation of the context early (superseded activation buffers / tensors set twice)
static void dev_free(ns_llama* c, void* p) {
  if (!p) return;
  for (size_t i = 0; i < c->owned.size(); ++i)
    if (c->owned[i] == p) {
      c->owned.erase(c->owned.begin() + (long)i);
      cudaFree(p);
      return;
    }
}

// the captured one-token graph bakes in pointers and the enqueued work: rebuilt at the next one-token eval
static void drop_decode_graph(ns_llama* c) {
  if (!c->decode_exec) return;
  cudaGraphExecDestroy(c->decode_exec);
  cudaGraphDestroy(c->decode_graph);
  c->decode_exec = nullptr;
  c->decode_graph = nullptr;
}

extern "C" ns_llama* ns_llama_create(const ns_llama_hparams* hp, void* queue) {
  if (ns_ensure_device()) return nullptr;
  if (!hp || hp->n_vocab <= 0 || hp->n_embd <= 0 || hp->n_head <= 0 || hp->n_head_kv <= 0 || hp->n_layer <= 0 || hp->n_ff <= 0 ||
      hp->n_ctx <= 0 || hp->n_embd % hp->n_head || hp->n_head % hp->n_head_kv || (hp->n_embd / hp->n_head) % 2 || hp->n_embd % 4) {
    ns_set_error("ns_llama_create: invalid hyper-parameters");
    return nullptr;
  }
  ns_llama* c = new ns_llama();
  c->hp = *hp;
  if (c->hp.rope_theta <= 0.f) c->hp.rope_theta = 10000.f;
  if (c->hp.rope_scale <= 0.f) c->hp.rope_scale = 1.f;
  if (c->hp.norm_eps <= 0.f) c->hp.norm_eps = 1e-6f;
  c->st = ns_stream_of(queue);
  c->layers.resize(hp->n_layer);
  const int hd = hp->n_embd / hp->n_head;
  {  // the single-pass attention kernels keep one score per cached position in shared memory
    const size_t need = (size_t)((3 + kAW) * hd + hp->n_ctx) * sizeof(float);
    if (need > 220 * 1024) {
      ns_set_error("ns_llama_create: n_ctx %d too large for the single-pass attention kernel (limit %zu positions at head size %d)",
                   hp->n_ctx, (size_t)(220 * 1024) / sizeof(float) - (size_t)(3 + kAW) * hd, hd);
      delete c;
      return nullptr;
    }
  }
  const size_t kv_elems = (size_t)hp->n_layer * hp->n_head_kv * hp->n_ctx * hd;
  c->kc = (__half*)dev_alloc(c, kv_elems * 2);
  c->vc = (__half*)dev_alloc(c, kv_elems * 2);
  c->state = (int*)dev_alloc(c, 4 * sizeof(int));
  c->tokens = (int*)dev_alloc(c, (size_t)hp->n_ctx * sizeof(int));
  c->record = (int*)dev_alloc(c, (size_t)hp->n_ctx * sizeof(int));
  c->logits = (float*)dev_alloc(c, (size_t)hp->n_vocab * 4);
  c->am_val = (float*)dev_alloc(c, 64 * sizeof(float));
  c->am_idx = (int*)dev_alloc(c, 64 * sizeof(int));
  c->am_ticket = (unsigned*)dev_alloc(c, sizeof(unsigned));
  if (c->am_ticket) cudaMemsetAsync(c->am_ticket, 0, sizeof(unsigned), c->st);
  c->attn_nsplit = (hp->n_ctx + kSplitKeys - 1) / kSplitKeys;
  c->attn_part = (float*)dev_alloc(c, (size_t)hp->n_head * c->attn_nsplit * (hd + 2) * sizeof(float));
  c->attn_tickets = (unsigned*)dev_alloc(c, (size_t)hp->n_head * sizeof(unsigned));
  if (c->attn_tickets) cudaMemsetAsync(c->attn_tickets, 0, (size_t)hp->n_head * sizeof(unsigned), c->st);
  if (!c->kc || !c->vc || !c->state || !c->tokens || !c->record || !c->logits || !c->am_val || !c->am_idx || !c->am_ticket ||
      !c->attn_part || !c->attn_tickets ||
      cudaMallocHost((void**)&c->h_state, 4 * sizeof(int)) != cudaSuccess ||
      cudaMallocHost((void**)&c->h_logits, (size_t)hp->n_vocab * 4) != cudaSuccess) {
    ns_llama_free(c);
    return nullptr;
  }
  cudaMemsetAsync(c->kc, 0, kv_elems * 2, c->st);
  cudaMemsetAsync(c->vc, 0, kv_elems * 2, c->st);
  cudaMemsetAsync(c->state, 0, 4 * sizeof(int), c->st);
  return c;
}

extern "C" void ns_llama_free(ns_llama* c) {
  if (!c) return;
  cudaStreamSynchronize(c->st);
  if (c->decode_exec) cudaGraphExecDestroy(c->decode_exec);
  if (c->decode_graph) cudaGraphDestroy(c->decode_graph);
  for (void* p : c->owned) cudaFree(p);
  if (c->h_state) cudaFreeHost(c->h_state);
  if (c->h_logits) cudaFreeHost(c->h_logits);
  delete c;
}

extern "C" int ns_llama_set_f32(ns_llama* c, int tensor, int layer, const float* host, size_t count) {
  if (!c || !host) return NS_E_INVALID;
  const ns_llama_hparams& hp = c->hp;
  size_t want = 0;
  if (tensor == NS_LT_TOK_EMBD) want = (size_t)hp.n_vocab * hp.n_embd;
  else if (tensor == NS_LT_OUT_NORM || tensor == NS_LT_ATTN_NORM || tensor == NS_LT_FFN_NORM) want = hp.n_embd;
  if (!want || count != want || ((tensor == NS_LT_ATTN_NORM || tensor == NS_LT_FFN_NORM) && (layer < 0 || layer >= hp.n_layer))) {
    ns_set_error("ns_llama_set_f32: tensor %d layer %d count %zu", tensor, layer, count);
    return NS_E_INVALID;
  }
  float* d = (float*)dev_alloc(c, want * 4);
  if (!d) return NS_E_CUDA;
  NS_CUDA_TRY(cudaMemcpyAsync(d, host, want * 4, cudaMemcpyHostToDevice, c->st));
  NS_CUDA_TRY(cudaStreamSynchronize(c->st));  // also: nothing in flight reads the tensor this call replaces
  const float** slot = tensor == NS_LT_TOK_EMBD   ? (const float**)&c->tok_embd
                       : tensor == NS_LT_OUT_NORM ? (const float**)&c->out_norm
                       : tensor == NS_LT_ATTN_NORM ? &c->layers[layer].attn_norm
                                                   : &c->layers[layer].ffn_norm;
  if (*slot) {  // set twice: the captured decode graph holds the old pointer
    drop_decode_graph(c);
    dev_free(c, (void*)*slot);
  }
  *slot = d;
  return NS_OK;
}

extern "C" int ns_llama_set_weight(ns_llama* c, int tensor, int layer, const ns_weight* w) {
  if (!c || !w) return NS_E_INVALID;
  const ns_llama_hparams& hp = c->hp;
  const int hd = hp.n_embd / hp.n_head, kvd = hd * hp.n_head_kv;
  int n = 0, k = hp.n_embd;
  switch (tensor) {
    case NS_LT_OUTPUT: n = hp.n_vocab; break;
    case NS_LT_WQ: n = hp.n_embd; break;
    case NS_LT_WK: case NS_LT_WV: n = kvd; break;
    case NS_LT_WO: n = hp.n_embd; break;
    case NS_LT_W1: case NS_LT_W3: n = hp.n_ff; break;
    case NS_LT_W2: n = hp.n_embd; k = hp.n_ff; break;
    default: n = 0;
  }
  if (!n || w->n != n || w->k != k || (tensor != NS_LT_OUTPUT && (layer < 0 || layer >= hp.n_layer))) {
    ns_set_error("ns_llama_set_weight: tensor %d layer %d wants %dx%d, got %dx%d", tensor, layer, n, k, w->n, w->k);
    return NS_E_INVALID;
  }
  if (tensor == NS_LT_OUTPUT) {
    c->output = w;
  } else {
    Layer& l = c->layers[layer];
    const ns_weight** slot = tensor == NS_LT_WQ ? &l.wq : tensor == NS_LT_WK ? &l.wk : tensor == NS_LT_WV ? &l.wv
                           : tensor == NS_LT_WO ? &l.wo : tensor == NS_LT_W1 ? &l.w1 : tensor == NS_LT_W2 ? &l.w2 : &l.w3;
    *slot = w;
  }
  drop_decode_graph(c);  // weights changed: the captured graph holds stale pointers
  return NS_OK;
}

static int launch_rmsnorm(const float* x, const float* w, float* y, int rows, int n, float eps, cudaStream_t st) {
  if (n % 4 || n > 256 * 4 * 8) {
    ns_set_error("ns_llama: n_embd %d unsupported by the RMSNorm kernel (needs n %% 4 == 0, n <= 8192)", n);
    return NS_E_UNSUPPORTED;
  }
  const int v4 = (n / 4 + 255) / 256;
  auto kern = v4 <= 1 ? rmsnorm_kernel<1> : v4 <= 2 ? rmsnorm_kernel<2> : v4 <= 4 ? rmsnorm_kernel<4> : rmsnorm_kernel<8>;
  NS_CUDA_TRY(ns_launch_pdl(kern, dim3((unsigned)rows), dim3(256), 0, st, x, w, y, n, eps));
  ns_count_launch();
  return NS_OK;
}

static int ensure_buffers(ns_llama* c, int m) {
  if (m <= c->m_cap) return NS_OK;
  const ns_llama_hparams& hp = c->hp;
  const int hd = hp.n_embd / hp.n_head, kvd = hd * hp.n_head_kv;
  if (c->m_cap > 0) {  // growing: the smaller buffers are dead once the stream has drained
    NS_CUDA_TRY(cudaStreamSynchronize(c->st));
    void* old[6] = {c->x, c->xn, c->qkv, c->attn, c->tmp, c->ws};
    for (void* p : old) dev_free(c, p);
    c->x = c->xn = c->qkv = c->attn = c->tmp = nullptr;
    c->ws = nullptr;
    c->m_cap = 0;
  }
  c->x = (float*)dev_alloc(c, (size_t)m * hp.n_embd * 4);
  c->xn = (float*)dev_alloc(c, (size_t)m * hp.n_embd * 4);
  c->qkv = (float*)dev_alloc(c, (size_t)m * (hp.n_embd + 2 * kvd) * 4);
  c->attn = (float*)dev_alloc(c, (size_t)m * hp.n_embd * 4);
  c->tmp = (float*)dev_alloc(c, (size_t)2 * m * hp.n_ff * 4);
  const int kmax = hp.n_ff > hp.n_embd ? hp.n_ff : hp.n_embd;
  size_t wsb = ns_act_workspace_bytes(4, (int)ns_round_up((size_t)kmax, 32));
  const size_t tcb = ns_gemm_tc_workspace_bytes(m, (int)ns_round_up((size_t)kmax, 32));
  const size_t q6 = ns_q6k_workspace_bytes(4, kmax);
  const size_t imb = ns_gemm_imma_workspace_bound(m > 32 ? 32 : (m < 5 ? 5 : m), (int)ns_round_up((size_t)kmax, 32));
  wsb = wsb > tcb ? wsb : tcb;
  wsb = wsb > q6 ? wsb : q6;
  wsb = wsb > imb ? wsb : imb;
  c->ws = dev_alloc(c, wsb);
  c->ws_bytes = wsb;
  if (!c->x || !c->xn || !c->qkv || !c->attn || !c->tmp || !c->ws) return NS_E_CUDA;
  c->m_cap = m;
  drop_decode_graph(c);
  return NS_OK;
}

static int check_complete(const ns_llama* c) {
  if (!c->tok_embd || !c->out_norm || !c->output) {
    ns_set_error("ns_llama: tok_embeddings / output norm / output weight not set");
    return NS_E_INVALID;
  }
  for (size_t i = 0; i < c->layers.size(); ++i) {
    const Layer& l = c->layers[i];
    if (!l.attn_norm || !l.ffn_norm || !l.wq || !l.wk || !l.wv || !l.wo || !l.w1 || !l.w2 || !l.w3) {
      ns_set_error("ns_llama: layer %zu is missing tensors", i);
      return NS_E_INVALID;
    }
  }
  return NS_OK;
}

// enqueue the whole forward pass for m new tokens (ids in c->tokens[0..m) or, when from_state, the single id in
// state[0]); position base = state[1].  Leaves logits of the LAST token in c->logits and the greedy pick in state[3].
static int enqueue_forward(ns_llama* c, int m, bool from_state, int advance, int* record) {
  const ns_llama_hparams& hp = c->hp;
  cudaStream_t st = c->st;
  const int E = hp.n_embd, hd = E / hp.n_head, kvd = hd * hp.n_head_kv, FF = hp.n_ff;
  const float theta_scale = powf(hp.rope_theta, -2.0f / (float)hd);  // n_rot == head_size (llama.cpp:131)
  const float freq_scale = 1.f / hp.rope_scale;
  const float attn_scale = 1.0f / sqrtf((float)hd);
  float* q = c->qkv;
  float* k = q + (size_t)m * E;
  float* v = k + (size_t)m * kvd;
  NS_CUDA_TRY(ns_launch_pdl(embed_kernel, dim3((unsigned)((E / 4 + 255) / 256), (unsigned)m), dim3(256), 0, st, (const float*)c->tok_embd,
                            (const int*)(from_state ? c->state : c->tokens), E, hp.n_vocab, c->x));
  ns_count_launch();
  const size_t attn_smem = (size_t)(hd + hp.n_ctx) * sizeof(float);
  size_t& attn_attr = c->attn_attr;  // per context: the function attribute is per device
  if (attn_smem > 48 * 1024 && attn_smem > attn_attr) {
    if (attn_smem > 220 * 1024) {
      ns_set_error("ns_llama: n_ctx %d too large for the single-pass attention kernel", hp.n_ctx);
      return NS_E_UNSUPPORTED;
    }
    NS_CUDA_TRY(cudaFuncSetAttribute(attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_smem));
    attn_attr = attn_smem;
  }
  const size_t fast_smem = (size_t)((3 + kAW) * hd + hp.n_ctx) * sizeof(float);
  if (fast_smem > 48 * 1024) {
    size_t& fast_attr = c->fast_attr;
    if (fast_smem > 220 * 1024) {
      ns_set_error("ns_llama: n_ctx %d too large for the single-pass attention kernel", hp.n_ctx);
      return NS_E_UNSUPPORTED;
    }
    if (fast_smem > fast_attr) {
      NS_CUDA_TRY(cudaFuncSetAttribute(attn_fast_kernel<128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
      NS_CUDA_TRY(cudaFuncSetAttribute(attn_fast_kernel<128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
      NS_CUDA_TRY(cudaFuncSetAttribute(attn_fast_kernel<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
      NS_CUDA_TRY(cudaFuncSetAttribute(attn_fast_kernel<64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
      fast_attr = fast_smem;
    }
  }
  // debugging aids, read per eval (not per process) so that a test can compare kernels on one engine
  const bool old_decode = getenv("NS_ATTN_OLD_DECODE") != nullptr;  // decode attention: one CTA per head, dependent row loads
  const bool scalar_attn = getenv("NS_ATTN_SCALAR") != nullptr;    // prompt attention: one CTA per (head, token), no tensor cores
  for (int il = 0; il < hp.n_layer; ++il) {
    const Layer& L = c->layers[il];
    __half* kc = c->kc + (size_t)il * hp.n_head_kv * hp.n_ctx * hd;
    __half* vc = c->vc + (size_t)il * hp.n_head_kv * hp.n_ctx * hd;
    // Decode rows: the attention RMSNorm (llama.cpp:205-210) rides in the activation quantiser of the Q/K/V launch(es) -- every
    // CTA reads the whole row anyway -- instead of a one-CTA kernel and a launch boundary of its own.
    const ns_weight* qkvw[3] = {L.wq, L.wk, L.wv};
    bool fused = false;
    if (hp.n_head == hp.n_head_kv && ns_gemv_fused_norm_ok(qkvw, 3, m))
      fused = ns_mul_qkv_norm(L.wq, L.wk, L.wv, c->x, E, q, E, m, c->ws, (void*)st, L.attn_norm, hp.norm_eps) == NS_OK;
    if (!fused && hp.n_head != hp.n_head_kv && ns_gemv_fused_norm_ok(&qkvw[0], 1, m) && ns_gemv_fused_norm_ok(&qkvw[1], 1, m) &&
        ns_gemv_fused_norm_ok(&qkvw[2], 1, m)) {
      if (int rc = ns_rmsnorm_mul_mat(L.wq, c->x, E, L.attn_norm, hp.norm_eps, q, E, m, nullptr, c->ws, (void*)st)) return rc;
      if (int rc = ns_rmsnorm_mul_mat(L.wk, c->x, E, L.attn_norm, hp.norm_eps, k, kvd, m, nullptr, c->ws, (void*)st)) return rc;
      if (int rc = ns_rmsnorm_mul_mat(L.wv, c->x, E, L.attn_norm, hp.norm_eps, v, kvd, m, nullptr, c->ws, (void*)st)) return rc;
      fused = true;
    }
    if (!fused) {
      if (int rc = launch_rmsnorm(c->x, L.attn_norm, c->xn, m, E, hp.norm_eps, st)) return rc;
      if (hp.n_head == hp.n_head_kv) {  // fused QKV node (llama.cpp:212-215); dst = [3][m][E] = q | k | v
        fused = ns_mul_qkv(L.wq, L.wk, L.wv, c->xn, E, q, E, m, c->ws, (void*)st) == NS_OK;
      }
      if (!fused) {
        if (int rc = ns_mul_mat(L.wq, c->xn, E, q, E, m, nullptr, nullptr, 0, c->ws, (void*)st)) return rc;
        if (int rc = ns_mul_mat(L.wk, c->xn, E, k, kvd, m, nullptr, nullptr, 0, c->ws, (void*)st)) return rc;
        if (int rc = ns_mul_mat(L.wv, c->xn, E, v, kvd, m, nullptr, nullptr, 0, c->ws, (void*)st)) return rc;
      }
    }
    const bool tap = il == c->tap_layer;
    if (tap)  // before any RoPE: rope_kv_kernel rotates q in place
      NS_CUDA_TRY(cudaMemcpyAsync(c->tap_qkv, c->qkv, (size_t)m * (E + 2 * kvd) * 4, cudaMemcpyDeviceToDevice, st));
    const bool fast = (hd == 128 || hd == 64);
    static const int dbg_skip = getenv("NS_LLAMA_DEBUG_SKIP") ? atoi(getenv("NS_LLAMA_DEBUG_SKIP")) : 0;  // timing experiments only
    if (m == 1 && (dbg_skip & 1)) {
      // (results are wrong: the attention launch is left out to measure what it costs inside the token's graph)
    } else if (fast && m == 1 && c->attn_nsplit <= 1024 && !old_decode) {
      // rope + KV append + attention in one launch, K / V staged by TMA, the context split over CTAs
      const size_t dsm = hd == 128 ? attn_decode_smem<128>() : attn_decode_smem<64>();
      if (!c->dec_attr) {
        NS_CUDA_TRY(cudaFuncSetAttribute(attn_decode_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_decode_smem<128>()));
        NS_CUDA_TRY(cudaFuncSetAttribute(attn_decode_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_decode_smem<64>()));
        c->dec_attr = 1;
      }
      auto kern = hd == 128 ? attn_decode_kernel<128> : attn_decode_kernel<64>;
      NS_CUDA_TRY(ns_launch_pdl(kern, dim3((unsigned)hp.n_head, (unsigned)c->attn_nsplit), dim3(kDW * 32), dsm, st, (const float*)q,
                                (const float*)k, (const float*)v, kc, vc, (const int*)c->state, c->attn, c->attn_part, c->attn_tickets,
                                hp.n_head, hp.n_head_kv, hp.n_ctx, c->attn_nsplit, attn_scale, theta_scale, freq_scale));
      ns_count_launch();
    } else if (fast && m == 1) {  // the same fused launch with dependent row loads (one CTA per head)
      auto kern = hd == 128 ? attn_fast_kernel<128, true> : attn_fast_kernel<64, true>;
      NS_CUDA_TRY(ns_launch_pdl(kern, dim3((unsigned)hp.n_head, 1u), dim3(kAW * 32), fast_smem, st, (const float*)q, E, (const float*)k, kvd,
                                (const float*)v, kvd, kc, vc, (const int*)c->state, c->attn, E, hp.n_head, hp.n_head_kv, hp.n_ctx,
                                attn_scale, theta_scale, freq_scale));
      ns_count_launch();
    } else {
      NS_CUDA_TRY(ns_launch_pdl(rope_kv_kernel, dim3((unsigned)(hp.n_head + hp.n_head_kv), (unsigned)m), dim3((unsigned)(hd / 2)), 0, st, q,
                                E, (const float*)k, kvd, (const float*)v, kvd, kc, vc, (const int*)c->state, hp.n_head, hp.n_head_kv, hd,
                                hp.n_ctx, theta_scale, freq_scale));
      ns_count_launch();
      // prompts: causal attention on the tensor cores (64 query rows per CTA); a handful of rows stay on the decode-shaped kernel
      const bool mma = fast && m >= 8 && !(E % 2) && !scalar_attn;
      if (mma) {
        auto kern = hd == 128 ? attn_mma_kernel<128> : attn_mma_kernel<64>;
        NS_CUDA_TRY(ns_launch_pdl(kern, dim3((unsigned)((m + kAttnMmaRows - 1) / kAttnMmaRows), (unsigned)hp.n_head), dim3(128), 0, st,
                                  (const float*)q, E, (const __half*)kc, (const __half*)vc, (const int*)c->state, c->attn, E, hp.n_head,
                                  hp.n_head_kv, hp.n_ctx, m, attn_scale));
      } else if (fast) {
        auto kern = hd == 128 ? attn_fast_kernel<128, false> : attn_fast_kernel<64, false>;
        NS_CUDA_TRY(ns_launch_pdl(kern, dim3((unsigned)hp.n_head, (unsigned)m), dim3(kAW * 32), fast_smem, st, (const float*)q, E,
                                  (const float*)k, kvd, (const float*)v, kvd, kc, vc, (const int*)c->state, c->attn, E, hp.n_head,
                                  hp.n_head_kv, hp.n_ctx, attn_scale, theta_scale, freq_scale));
      } else {
        NS_CUDA_TRY(ns_launch_pdl(attn_kernel, dim3((unsigned)hp.n_head, (unsigned)m), dim3(kAttnThreads), attn_smem, st, (const float*)q,
                                  E, (const __half*)kc, (const __half*)vc, (const int*)c->state, c->attn, E, hp.n_head, hp.n_head_kv, hd,
                                  hp.n_ctx, attn_scale));
      }
      ns_count_launch();
    }
    if (tap) NS_CUDA_TRY(cudaMemcpyAsync(c->tap_attn, c->attn, (size_t)m * E * 4, cudaMemcpyDeviceToDevice, st));
    // inpFF = wo * attn + inpSA, written over x (every row is read by its own output only after the matmul finished)
    if (int rc = ns_mul_mat_engine(L.wo, c->attn, E, c->xn, E, m, c->x, c->ws, st, nullptr, 0.f)) return rc;
    // xn now holds inpFF; FFN + residual back into x, the FFN RMSNorm folded into the gate/up launch where that is a ring GEMV,
    // else normalised into attn (free again) first
    const ns_weight* guw[2] = {L.w1, L.w3};
    if (ns_gemv_fused_norm_ok(guw, 2, m)) {
      if (int rc = ns_ffn_silu_residual(L.w1, L.w2, L.w3, c->xn, E, c->tmp, c->x, E, m, c->xn, c->ws, st, L.ffn_norm, hp.norm_eps, 1)) return rc;
    } else {
      if (int rc = launch_rmsnorm(c->xn, L.ffn_norm, c->attn, m, E, hp.norm_eps, st)) return rc;
      if (int rc = ns_ffn_silu_residual(L.w1, L.w2, L.w3, c->attn, E, c->tmp, c->x, E, m, c->xn, c->ws, st, nullptr, 0.f, 1)) return rc;
    }
  }
  // logits of the last token only (model_eval keeps the last row unless logits_all)
  const ns_weight* outw[1] = {c->output};
  if (ns_gemv_fused_norm_ok(outw, 1, 1)) {
    if (int rc = ns_rmsnorm_mul_mat(c->output, c->x + (size_t)(m - 1) * E, E, c->out_norm, hp.norm_eps, c->logits, hp.n_vocab, 1, nullptr,
                                    c->ws, (void*)st))
      return rc;
  } else {
    if (int rc = launch_rmsnorm(c->x + (size_t)(m - 1) * E, c->out_norm, c->xn, 1, E, hp.norm_eps, st)) return rc;
    if (int rc = ns_mul_mat(c->output, c->xn, E, c->logits, hp.n_vocab, 1, nullptr, nullptr, 0, c->ws, (void*)st)) return rc;
  }
  NS_CUDA_TRY(ns_launch_pdl(argmax_kernel, dim3((unsigned)kArgmaxBlocks), dim3(256), 0, st, (const float*)c->logits, hp.n_vocab, c->state, m,
                            advance, record, c->am_val, c->am_idx, c->am_ticket));
  ns_count_launch();
  return NS_OK;
}

static int ensure_decode_graph(ns_llama* c) {
  if (c->decode_exec) return NS_OK;
  // one eager pass (no state advance; it writes the same K/V the real pass will) sets kernel attributes and sizes every
  // lazily-grown buffer outside the capture, then capture
  if (int rc = enqueue_forward(c, 1, true, 0, nullptr)) return rc;
  NS_CUDA_TRY(cudaStreamSynchronize(c->st));
  NS_CUDA_TRY(cudaStreamBeginCapture(c->st, cudaStreamCaptureModeThreadLocal));
  int rc = enqueue_forward(c, 1, true, 1, c->record);
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamEndCapture(c->st, &g);
  if (rc) {
    if (g) cudaGraphDestroy(g);
    return rc;
  }
  if (!ns_cuda_ok(e, "cudaStreamEndCapture") || !g) return NS_E_CUDA;
  if (!ns_cuda_ok(cudaGraphInstantiate(&c->decode_exec, g, 0), "cudaGraphInstantiate")) {
    cudaGraphDestroy(g);
    return NS_E_CUDA;
  }
  c->decode_graph = g;
  return NS_OK;
}

// model_eval (models/model_utils/model_utils.h): evaluate n_tokens new tokens after n_past cached ones.
// logits_host (nullable): n_vocab floats of the LAST token; next_token (nullable): its greedy pick.
extern "C" int ns_llama_set_exact_prefill(ns_llama* c, int on) {
  if (!c) return NS_E_INVALID;
  c->exact_prefill = on ? 1 : 0;
  return NS_OK;
}

extern "C" int ns_llama_eval(ns_llama* c, const int32_t* tokens, int n_tokens, int n_past, float* logits_host, int32_t* next_token) {
  if (int rc = ns_ensure_device()) return rc;
  if (!c || !tokens || n_tokens <= 0 || n_past < 0 || n_past + n_tokens > c->hp.n_ctx) {
    ns_set_error("ns_llama_eval: invalid arguments (n_tokens=%d n_past=%d n_ctx=%d)", n_tokens, n_past, c ? c->hp.n_ctx : 0);
    return NS_E_INVALID;
  }
  if (c->tap_layer >= 0 && n_tokens > c->tap_rows) {
    ns_set_error("ns_llama_eval: %d new tokens, the tap set with ns_llama_set_tap holds %d rows", n_tokens, c->tap_rows);
    return NS_E_INVALID;
  }
  if (c->exact_prefill && n_tokens > 32) {
    // parity mode: prompts go through in pieces of <= 32 tokens, which the matmuls run on the integer tensor cores with the
    // reference's exact block sums (causal attention over the fp16 KV cache makes the split invisible to the arithmetic)
    for (int t0 = 0; t0 < n_tokens; t0 += 32) {
      const int nt = n_tokens - t0 < 32 ? n_tokens - t0 : 32;
      const bool last = t0 + nt == n_tokens;
      if (int rc = ns_llama_eval(c, tokens + t0, nt, n_past + t0, last ? logits_host : nullptr, last ? next_token : nullptr)) return rc;
    }
    return NS_OK;
  }
  if (int rc = check_complete(c)) return rc;
  if (int rc = ensure_buffers(c, n_tokens)) return rc;
  cudaStream_t st = c->st;
  c->h_state[0] = tokens[0];
  c->h_state[1] = n_past;
  c->h_state[2] = 0;
  c->h_state[3] = 0;
  NS_CUDA_TRY(cudaMemcpyAsync(c->state, c->h_state, 4 * sizeof(int), cudaMemcpyHostToDevice, st));
  if (n_tokens == 1) {
    if (int rc = ensure_decode_graph(c)) return rc;
    NS_CUDA_TRY(cudaGraphLaunch(c->decode_exec, st));
  } else {
    NS_CUDA_TRY(cudaMemcpyAsync(c->tokens, tokens, (size_t)n_tokens * sizeof(int), cudaMemcpyHostToDevice, st));
    if (int rc = enqueue_forward(c, n_tokens, false, 1, nullptr)) return rc;
  }
  if (logits_host) NS_CUDA_TRY(cudaMemcpyAsync(c->h_logits, c->logits, (size_t)c->hp.n_vocab * 4, cudaMemcpyDeviceToHost, st));
  NS_CUDA_TRY(cudaMemcpyAsync(c->h_state, c->state, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
  NS_CUDA_TRY(cudaStreamSynchronize(st));
  if (logits_host) memcpy(logits_host, c->h_logits, (size_t)c->hp.n_vocab * 4);
  if (next_token) *next_token = c->h_state[3];
  return NS_OK;
}

// greedy generation: token `first` at position n_past, then n_new - 1 more, each fed from the previous argmax on the
// device (one graph launch per token, no host synchronisation in between).  out_tokens[i] = pick after step i.
extern "C" int ns_llama_generate(ns_llama* c, int32_t first_token, int n_past, int n_new, int32_t* out_tokens) {
  if (int rc = ns_ensure_device()) return rc;
  if (!c || !out_tokens || n_new <= 0 || n_past < 0 || n_past + n_new > c->hp.n_ctx) {
    ns_set_error("ns_llama_generate: invalid arguments (n_past=%d n_new=%d n_ctx=%d)", n_past, n_new, c ? c->hp.n_ctx : 0);
    return NS_E_INVALID;
  }
  if (int rc = check_complete(c)) return rc;
  if (int rc = ensure_buffers(c, 1)) return rc;
  if (int rc = ensure_decode_graph(c)) return rc;
  cudaStream_t st = c->st;
  c->h_state[0] = first_token;
  c->h_state[1] = n_past;
  c->h_state[2] = 0;
  c->h_state[3] = 0;
  NS_CUDA_TRY(cudaMemcpyAsync(c->state, c->h_state, 4 * sizeof(int), cudaMemcpyHostToDevice, st));
  for (int i = 0; i < n_new; ++i) NS_CUDA_TRY(cudaGraphLaunch(c->decode_exec, st));
  NS_CUDA_TRY(cudaMemcpyAsync(out_tokens, c->record, (size_t)n_new * sizeof(int), cudaMemcpyDeviceToHost, st));
  NS_CUDA_TRY(cudaStreamSynchronize(st));
  return NS_OK;
}

extern "C" int ns_llama_set_tap(ns_llama* c, int layer, float* qkv_dst, float* attn_dst, int max_rows) {
  if (!c) return NS_E_INVALID;
  if (layer >= 0 && (layer >= c->hp.n_layer || !qkv_dst || !attn_dst || max_rows <= 0)) {
    ns_set_error("ns_llama_set_tap: layer %d of %d, max_rows %d", layer, c->hp.n_layer, max_rows);
    return NS_E_INVALID;
  }
  NS_CUDA_TRY(cudaStreamSynchronize(c->st));  // nothing in flight still writes to the previous destinations
  c->tap_layer = layer < 0 ? -1 : layer;
  c->tap_qkv = layer < 0 ? nullptr : qkv_dst;
  c->tap_attn = layer < 0 ? nullptr : attn_dst;
  c->tap_rows = layer < 0 ? 0 : max_rows;
  drop_decode_graph(c);  // the copies are (or were) nodes of the captured graph
  return NS_OK;
}

extern "C" int ns_llama_kv_cache(const ns_llama* c, int layer, const void** k, const void** v) {
  if (!c || !k || !v || layer < 0 || layer >= c->hp.n_layer) {
    ns_set_error("ns_llama_kv_cache: invalid arguments (layer %d)", layer);
    return NS_E_INVALID;
  }
  const size_t per_layer = (size_t)c->hp.n_head_kv * c->hp.n_ctx * (c->hp.n_embd / c->hp.n_head);
  *k = c->kc + (size_t)layer * per_layer;
  *v = c->vc + (size_t)layer * per_layer;
  return NS_OK;
}

extern "C" unsigned long long ns_llama_kv_bytes(const ns_llama* c) {
  if (!c) return 0;
  return (unsigned long long)2 * c->hp.n_layer * c->hp.n_head_kv * c->hp.n_ctx * (c->hp.n_embd / c->hp.n_head) * 2;
}
