// Bandwidth-bound / small-contraction kernels (plain SIMT, fp32): stem conv, fp32->split-fp16 conversion,
// linear-attention state reduction and application, dual-softmax statistics merge, mutual-NN selection.
#pragma once
#include "tc_common.cuh"

namespace dfsfm {

// --------------------------------------------------------------------------------------------------------
// 7x7 stride-2 pad-3 convolution 1 -> 128 channels + folded BN + ReLU  (ResNetFPN_8_2.conv1/bn1/relu,
// third_party/LoFTR/src/loftr/backbone/resnet_fpn.py:100-102).  Output: flat-halo split-fp16, pitch W/2+1, image n = blockIdx.z
// (img0 or img1) at flat block n.  CTA = 8x16 output pixels, thread = output channel.
constexpr int kStemTH = 8, kStemTW = 16;
static __global__ void __launch_bounds__(128) stem_conv_kernel(const float* __restrict__ img0, const float* __restrict__ img1, int H, int W,
                                                        const float* __restrict__ w /*[128][49]*/, const float* __restrict__ bias,
                                                        __half* __restrict__ out_hi, __half* __restrict__ out_lo) {
    constexpr int IH = kStemTH * 2 + 5, IW = kStemTW * 2 + 5;
    constexpr int PITCH = 40;  // 16-byte aligned rows: a thread reads 16 consecutive inputs as 4 x float4 for 4 output pixels
    __shared__ __align__(16) float tile[IH][PITCH];
    const int H2 = H / 2, W2 = W / 2, Wp = W2 + 1;
    const int oy0 = blockIdx.y * kStemTH, ox0 = blockIdx.x * kStemTW;
    const int n = blockIdx.z;
    const float* im = n == 0 ? img0 : img1;
    for (int i = threadIdx.x; i < IH * PITCH; i += 128) {
        const int ty = i / PITCH, tx = i - ty * PITCH;
        const int iy = oy0 * 2 - 3 + ty, ix = ox0 * 2 - 3 + tx;
        tile[ty][tx] = (tx < IW && iy >= 0 && iy < H && ix >= 0 && ix < W) ? im[static_cast<long long>(iy) * W + ix] : 0.f;
    }
    const int c = threadIdx.x;
    float wr[49];
#pragma unroll
    for (int i = 0; i < 49; ++i) wr[i] = w[c * 49 + i];
    const float b = bias[c];
    __syncthreads();
    const long long img_rows = static_cast<long long>(H2 + 1) * Wp;
    for (int py = 0; py < kStemTH; ++py) {
        const int oy = oy0 + py;
        if (oy >= H2) break;
#pragma unroll 1
        for (int pg = 0; pg < kStemTW / 4; ++pg) {  // 4 adjacent output pixels per pass share their input rows
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int ky = 0; ky < 7; ++ky) {
                float in[16];
                const float4* rp = reinterpret_cast<const float4*>(&tile[py * 2 + ky][pg * 8]);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 v = rp[q];
                    in[4 * q] = v.x; in[4 * q + 1] = v.y; in[4 * q + 2] = v.z; in[4 * q + 3] = v.w;
                }
#pragma unroll
                for (int p = 0; p < 4; ++p)
#pragma unroll
                    for (int kx = 0; kx < 7; ++kx) acc[p] = fmaf(wr[ky * 7 + kx], in[2 * p + kx], acc[p]);
            }
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const int ox = ox0 + pg * 4 + p;
                if (ox < W2) {
                    const float r = fmaxf(acc[p] + b, 0.f);
                    const long long o = (n * img_rows + static_cast<long long>(oy) * Wp + ox) * 128 + c;
                    __half h, l;
                    split_f16(r, h, l);
                    out_hi[o] = h;
                    out_lo[o] = l;
                }
            }
        }
    }
}

// fp32 [rows][C] -> split-fp16 planes [rows][C]; C % 4 == 0.
static __global__ void split_rows_kernel(const float* __restrict__ in, long long n4, __half* __restrict__ hi, __half* __restrict__ lo) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i >= n4) return;
    const float4 v = reinterpret_cast<const float4*>(in)[i];
    __half h[4], l[4];
    split_f16(v.x, h[0], l[0]);
    split_f16(v.y, h[1], l[1]);
    split_f16(v.z, h[2], l[2]);
    split_f16(v.w, h[3], l[3]);
    reinterpret_cast<uint2*>(hi)[i] = *reinterpret_cast<uint2*>(h);
    reinterpret_cast<uint2*>(lo)[i] = *reinterpret_cast<uint2*>(l);
}

// --------------------------------------------------------------------------------------------------------
// Linear attention (third_party/LoFTR/src/loftr/loftr_module/linear_attention.py:20-47, identical maths in
// src/MultiviewMatcher/matcher_module/linear_attention.py:28-60).  K has already been through elu+1 (GEMM epilogue).
//   KV[h][d][v] = sum_s K[s,h,d] * (V[s,h,v] / len),  Ksum[h][d] = sum_s K[s,h,d]        (masked tokens skipped)
//   out[l,h,v]  = (sum_d Q[l,h,d] KV[h][d][v]) * (1 / (sum_d Q[l,h,d] Ksum[h][d] + eps)) * len
// A "segment" is one attention batch element (the whole image for HP-1, one track for HP-2).
struct Seg {
    int start;  // first token row
    int count;  // tokens in the segment (incl. masked ones: `len` of the reference is the padded length)
    int valid;  // leading tokens that are valid (kv_mask / q_mask); the rest are skipped
    int state;  // index of the KV state this segment writes / reads
};

constexpr int kKvTokPerCta = 64;
// grid (chunks, segments); block = 8 heads * D threads.  part: [seg][chunk][8*D*(D+1)].
// 16-token sub-batches: float4 global loads are issued one sub-batch ahead (register prefetch) so that the
// shared-memory outer-product loop of batch i runs under the loads of batch i+1.
template <int D>
static __global__ void __launch_bounds__(8 * D) kv_partial_kernel(const float* __restrict__ K, const float* __restrict__ V, int ld,
                                                            const Seg* __restrict__ segs, int max_chunks, float* __restrict__ part,
                                                            int tok_per_cta) {
    constexpr int C = 8 * D;
    constexpr int C4 = C / 4;
    constexpr int SUB = 16;
    // one buffer: the K / V staging tiles during the reduction, then the [C][D+1] result for a coalesced write-out
    constexpr int kBuf = C * (D + 1) > 2 * SUB * C ? C * (D + 1) : 2 * SUB * C;
    __shared__ __align__(16) float buf[kBuf];
    float (*Ks)[C] = reinterpret_cast<float (*)[C]>(buf);
    float (*Vs)[C] = reinterpret_cast<float (*)[C]>(buf + SUB * C);
    const Seg sg = segs[blockIdx.y];
    const int tid = threadIdx.x;
    const int h = tid / D;
    float acc[D];
#pragma unroll
    for (int v = 0; v < D; ++v) acc[v] = 0.f;
    float ksum = 0.f;
    const float len = static_cast<float>(sg.count);
    const int t0 = blockIdx.x * tok_per_cta;
    const int t1 = min(t0 + tok_per_cta, sg.valid);
    const int s0 = tid / C4, c4 = tid - s0 * C4;  // this thread stages tokens s0, s0+4, s0+8, s0+12 at columns [4*c4, 4*c4+4)
    float4 rk[4], rv[4];
    auto load = [&](int tb) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int t = tb + s0 + 4 * j;
            if (t < t1) {
                const long long r = static_cast<long long>(sg.start + t) * ld + c4 * 4;
                rk[j] = *reinterpret_cast<const float4*>(K + r);
                rv[j] = *reinterpret_cast<const float4*>(V + r);
            } else {
                rk[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                rv[j] = rk[j];
            }
        }
    };
    if (t0 < t1) load(t0);
    for (int tb = t0; tb < t1; tb += SUB) {
        const int nt = min(SUB, t1 - tb);
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            *reinterpret_cast<float4*>(&Ks[s0 + 4 * j][c4 * 4]) = rk[j];
            *reinterpret_cast<float4*>(&Vs[s0 + 4 * j][c4 * 4]) = make_float4(rv[j].x / len, rv[j].y / len, rv[j].z / len, rv[j].w / len);
        }
        __syncthreads();
        if (tb + SUB < t1) load(tb + SUB);
        for (int s = 0; s < nt; ++s) {
            const float k = Ks[s][tid];
            ksum += k;
            const float4* vp = reinterpret_cast<const float4*>(&Vs[s][h * D]);
#pragma unroll
            for (int v4 = 0; v4 < D / 4; ++v4) {
                const float4 vv = vp[v4];
                acc[4 * v4] = fmaf(k, vv.x, acc[4 * v4]);
                acc[4 * v4 + 1] = fmaf(k, vv.y, acc[4 * v4 + 1]);
                acc[4 * v4 + 2] = fmaf(k, vv.z, acc[4 * v4 + 2]);
                acc[4 * v4 + 3] = fmaf(k, vv.w, acc[4 * v4 + 3]);
            }
        }
    }
    __syncthreads();  // every thread is done reading the staging tiles
#pragma unroll
    for (int v = 0; v < D; ++v) buf[tid * (D + 1) + v] = acc[v];  // stride D+1: conflict-free
    buf[tid * (D + 1) + D] = ksum;
    __syncthreads();
    float* o = part + (static_cast<long long>(blockIdx.y) * max_chunks + blockIdx.x) * (C * (D + 1));
    for (int i = tid; i < C * (D + 1); i += C) o[i] = buf[i];  // coalesced
}
// state[seg.state][8*D*(D+1)] = sum over chunks in a fixed order (deterministic).  grid (ceil(SZ/64), segments); block
// (64 outputs x 4 chunk groups): each group sums every 4th chunk, the 4 partial sums are combined through shared memory.
constexpr int kKvFinalThreads = 256;
template <int D>
static __global__ void __launch_bounds__(kKvFinalThreads) kv_final_kernel(const float* __restrict__ part, const Seg* __restrict__ segs,
                                                                          int max_chunks, float* __restrict__ state, int tok_per_cta) {
    constexpr int SZ = 8 * D * (D + 1);
    __shared__ float red[4][64];
    const Seg sg = segs[blockIdx.y];
    const int nch = (sg.valid + tok_per_cta - 1) / tok_per_cta;
    const int li = threadIdx.x & 63, grp = threadIdx.x >> 6;
    const int i = blockIdx.x * 64 + li;
    float s = 0.f;
    if (i < SZ) {
        const float* p = part + static_cast<long long>(blockIdx.y) * max_chunks * SZ + i;
        int c = grp;
        for (; c + 12 < nch; c += 16) {
            const float v0 = p[static_cast<long long>(c) * SZ], v1 = p[static_cast<long long>(c + 4) * SZ];
            const float v2 = p[static_cast<long long>(c + 8) * SZ], v3 = p[static_cast<long long>(c + 12) * SZ];
            s += v0; s += v1; s += v2; s += v3;
        }
        for (; c < nch; c += 4) s += p[static_cast<long long>(c) * SZ];
    }
    red[grp][li] = s;
    __syncthreads();
    if (grp == 0 && i < SZ) state[static_cast<long long>(sg.state) * SZ + i] = (red[0][li] + red[1][li]) + (red[2][li] + red[3][li]);
}
// grid (token blocks of 32, segments); block 256 = 8 warps x 4 tokens.  lane + 32 j -> output channel (head, v).
// The warp's 4 query rows are staged in shared memory (coalesced float4 loads issued up front) and read back as broadcast
// float4 -- per 16 FMAs the inner loop issues 4 state loads + 4 query loads instead of 16 + 16 shuffles.
// Masked query tokens (index >= seg.valid) produce 0 (the reference multiplies Q by the mask).
// tokens per CTA (a multiple of 32): the KV state is loaded once per CTA; few big segments (HP-1) want many small CTAs,
// thousands of short segments (HP-2) want the state load amortised.
constexpr int kAttnTokCoarse = 32, kAttnTokRefine = 128;
template <int D>
constexpr int attn_smem_bytes() { return (8 * D * (D + 1) + 8 * 4 * 8 * D) * static_cast<int>(sizeof(float)); }
template <int D>
static __global__ void __launch_bounds__(256) attn_apply_kernel(const float* __restrict__ Q, int ldq, const Seg* __restrict__ segs,
                                                          const float* __restrict__ state, __half* __restrict__ out_hi,
                                                          __half* __restrict__ out_lo, int ldo, int tok_per_cta) {
    constexpr int C = 8 * D;
    constexpr int SZ = C * (D + 1);
    constexpr int NJ = C / 32;  // output channels per lane
    constexpr int TPW = 4;
    extern __shared__ __align__(16) float attn_sm[];
    float* st = attn_sm;             // [C][D+1]: KV[h][d][v] at (h*D+d)*(D+1)+v, Ksum at +D
    float* qs = attn_sm + SZ;        // [8 warps][TPW][C]
    const Seg sg = segs[blockIdx.y];
    if (blockIdx.x * tok_per_cta >= sg.count) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* qw = qs + warp * TPW * C;
    for (int i = threadIdx.x; i < SZ; i += 256) st[i] = state[static_cast<long long>(sg.state) * SZ + i];
    __syncthreads();
    const int hs = lane / D, v = lane - hs * D;  // D == 32: hs = 0, v = lane
    const float len = static_cast<float>(sg.count);
#pragma unroll 1
    for (int rep = 0; rep < tok_per_cta / (8 * TPW); ++rep) {
    const int tw = blockIdx.x * tok_per_cta + (rep * 8 + warp) * TPW;
    if (tw >= sg.count) break;
    __syncwarp();
    {   // stage this warp's query rows (zeros for masked / out-of-range tokens)
        constexpr int F4 = TPW * C / 4;
        for (int i = lane; i < F4; i += 32) {
            const int ti = i / (C / 4), c4 = i - ti * (C / 4);
            const int t = tw + ti;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (t < sg.valid) v = *reinterpret_cast<const float4*>(Q + static_cast<long long>(sg.start + t) * ldq + c4 * 4);
            *reinterpret_cast<float4*>(qw + ti * C + c4 * 4) = v;
        }
    }
    __syncwarp();
#pragma unroll 1
    for (int j = 0; j < NJ; ++j) {
        const int h = (32 * j) / D + hs;
        float acc[TPW], z[TPW];
#pragma unroll
        for (int ti = 0; ti < TPW; ++ti) { acc[ti] = 0.f; z[ti] = 0.f; }
        const float* kvh = st + (h * D) * (D + 1);
#pragma unroll
        for (int d4 = 0; d4 < D / 4; ++d4) {
            float kv[4], ks[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                kv[i] = kvh[(4 * d4 + i) * (D + 1) + v];
                ks[i] = kvh[(4 * d4 + i) * (D + 1) + D];
            }
#pragma unroll
            for (int ti = 0; ti < TPW; ++ti) {
                const float4 q4 = *reinterpret_cast<const float4*>(qw + ti * C + h * D + 4 * d4);
                acc[ti] = fmaf(q4.x, kv[0], acc[ti]); acc[ti] = fmaf(q4.y, kv[1], acc[ti]);
                acc[ti] = fmaf(q4.z, kv[2], acc[ti]); acc[ti] = fmaf(q4.w, kv[3], acc[ti]);
                z[ti] = fmaf(q4.x, ks[0], z[ti]); z[ti] = fmaf(q4.y, ks[1], z[ti]);
                z[ti] = fmaf(q4.z, ks[2], z[ti]); z[ti] = fmaf(q4.w, ks[3], z[ti]);
            }
        }
#pragma unroll
        for (int ti = 0; ti < TPW; ++ti) {
            const int t = tw + ti;
            if (t < sg.count) {
                const float r = acc[ti] * (1.f / (z[ti] + 1e-6f)) * len;
                __half hh, ll;
                split_f16(r, hh, ll);
                const long long o = static_cast<long long>(sg.start + t) * ldo + h * D + v;
                out_hi[o] = hh;
                out_lo[o] = ll;
            }
        }
    }
    }  // rep
}

// Sum the per-CTA partial states written by KvEpi (gemm_engine.cuh) in CTA order (deterministic) into the state layout the other
// kernels use: state[seg.state][(h*32+d)*33 + v], Ksum at v == 32; V's 1/len of linear_attention.py:39 is applied here.
// grid (ceil(8*32*33 / 64), launch segments), block 256 = 64 outputs x 4 CTA groups.
static __global__ void __launch_bounds__(256) kv_state_final_kernel(const float* __restrict__ part, const unsigned* __restrict__ flags, unsigned epoch,
                                                                    int n_ctas, int part_floats, const Seg* __restrict__ segs,
                                                                    float* __restrict__ state) {
    constexpr int SZ = 8 * 32 * 33, HS = 32 * 33;
    __shared__ float red[4][64];
    const int seg = blockIdx.y;
    const Seg sg = segs[seg];
    const int li = threadIdx.x & 63, grp = threadIdx.x >> 6;
    const int i = blockIdx.x * 64 + li;
    float s = 0.f;
    if (i < SZ) {
        const int h = i / HS, rem = i - h * HS;
        const int nt = h >> 2, hh = h & 3;
        const long long slot0 = static_cast<long long>(seg * 2 + nt) * n_ctas;
        const float* b = part + slot0 * part_floats + hh * HS + rem;
        const unsigned* f = flags + slot0;
        for (int c = grp; c < n_ctas; c += 4)
            if (f[c] == epoch) s += b[static_cast<long long>(c) * part_floats];
    }
    red[grp][li] = s;
    __syncthreads();
    if (grp == 0 && i < SZ) {
        const float t = (red[0][li] + red[1][li]) + (red[2][li] + red[3][li]);
        state[static_cast<long long>(sg.state) * SZ + i] = (i % 33) < 32 ? t / static_cast<float>(sg.count) : t;
    }
}

// Fold the attention state into the merge projection (HP-1 coarse layers, where a whole image shares one state):
//   message = merge( (Q*Z) . KV * len )  ==  (Q*Z*len) . G^T   with   G[n][h*D+d] = sum_v KV[h][d][v] * Wm[n][h*D+v]
// so that linear attention + merge (transformer.py:47-48, linear_attention.py:42-45) is ONE 256x256 GEMM per token tile against a
// per-call matrix, and neither q nor the message ever visit HBM as fp32.  grid (8 heads, segments), block 8*D (thread = output
// channel n).  `segs[i].state` picks the KV state, `.count` is the source length (v_length).  Also emits Ksum as a dense vector.
template <int D>
static __global__ void __launch_bounds__(8 * D) attn_fold_merge_kernel(const float* __restrict__ state, const Seg* __restrict__ segs,
                                                                       const __half* __restrict__ wm_hi, const __half* __restrict__ wm_lo,
                                                                       __half* __restrict__ g_hi, __half* __restrict__ g_lo,
                                                                       float* __restrict__ ksum_out) {
    constexpr int C = 8 * D;
    constexpr int SZ = C * (D + 1);
    __shared__ float kv[D][D + 1];
    const int h = blockIdx.x, seg = blockIdx.y, n = threadIdx.x;
    const Seg sg = segs[seg];
    const float* st = state + static_cast<long long>(sg.state) * SZ + (h * D) * (D + 1);
    for (int i = threadIdx.x; i < D * (D + 1); i += C) kv[i / (D + 1)][i % (D + 1)] = st[i];
    float w[D];
#pragma unroll
    for (int v = 0; v < D; v += 8) {
        const uint4 uh = *reinterpret_cast<const uint4*>(wm_hi + static_cast<long long>(n) * C + h * D + v);
        const uint4 ul = *reinterpret_cast<const uint4*>(wm_lo + static_cast<long long>(n) * C + h * D + v);
        const __half2* hh = reinterpret_cast<const __half2*>(&uh);
        const __half2* hl = reinterpret_cast<const __half2*>(&ul);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float2 a = __half22float2(hh[q]), b = __half22float2(hl[q]);
            w[v + 2 * q] = a.x + b.x;
            w[v + 2 * q + 1] = a.y + b.y;
        }
    }
    __syncthreads();
    if (n < D) ksum_out[seg * C + h * D + n] = kv[n][D];
    const long long o = (static_cast<long long>(seg) * C + n) * C + h * D;
#pragma unroll
    for (int d0 = 0; d0 < D; d0 += 8) {
        uint4 uh, ul;
        uint32_t* ph = reinterpret_cast<uint32_t*>(&uh);
        uint32_t* pl = reinterpret_cast<uint32_t*>(&ul);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int v = 0; v < D; ++v) {
                a0 = fmaf(kv[d0 + 2 * q][v], w[v], a0);
                a1 = fmaf(kv[d0 + 2 * q + 1][v], w[v], a1);
            }
            split_f16x2(a0, a1, ph[q], pl[q]);
        }
        *reinterpret_cast<uint4*>(g_hi + o + d0) = uh;
        *reinterpret_cast<uint4*>(g_lo + o + d0) = ul;
    }
}

// The same fold fed directly by the per-CTA partial states of KvEpi: one kernel sums the partials in CTA order (deterministic),
// applies V's 1/len, and writes G and Ksum -- the state itself never goes back to HBM.  Latency-bound (5 MB of partials per segment,
// a chain of dependent loads per thread), hence spread wide: grid (8 heads, 8 d-slices of 4 rows, launch segments) = 128 blocks for a
// pair, block 1024 = 7 CTA groups x 132 state elements for the sum, then 256 output channels x 4 d rows for the fold.
static __global__ void __launch_bounds__(1024) kvp_fold_kernel(const float* __restrict__ part, const unsigned* __restrict__ flags, unsigned epoch,
                                                               int n_ctas, const Seg* __restrict__ segs, const __half* __restrict__ wm_hi,
                                                               const __half* __restrict__ wm_lo, __half* __restrict__ g_hi, __half* __restrict__ g_lo,
                                                               float* __restrict__ ksum_out) {
    constexpr int D = 32, C = 256, HS = D * (D + 1), PF = 4 * HS, E = 4 * (D + 1), G = 7;
    __shared__ float red[G][E];
    __shared__ float kv[4][D + 1];
    __shared__ unsigned char ok[160];
    const int h = blockIdx.x, ds = blockIdx.y, seg = blockIdx.z, tid = threadIdx.x;
    const Seg sg = segs[seg];
    const int nt = h >> 2, hh = h & 3;
    const long long slot0 = static_cast<long long>(seg * 2 + nt) * n_ctas;
    for (int c = tid; c < n_ctas; c += 1024) ok[c] = flags[slot0 + c] == epoch;
    __syncthreads();
    const int grp = tid / E, e = tid - grp * E;
    if (grp < G) {
        const float* base = part + slot0 * PF + hh * HS + ds * E + e;   // rows d = 4*ds .. 4*ds+3 of head h: E consecutive floats
        float s = 0.f;
#pragma unroll 8
        for (int c = grp; c < n_ctas; c += G)
            if (ok[c]) s += base[static_cast<long long>(c) * PF];
        red[grp][e] = s;
    }
    __syncthreads();
    if (tid < E) {
        float v = red[0][tid];
#pragma unroll
        for (int g = 1; g < G; ++g) v += red[g][tid];
        (&kv[0][0])[tid] = (tid % (D + 1)) < D ? v / static_cast<float>(sg.count) : v;
    }
    __syncthreads();
    if (tid < 4) ksum_out[seg * C + h * D + ds * 4 + tid] = kv[tid][D];
    if (tid >= C) return;
    const int n = tid;
    float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int v = 0; v < D; v += 8) {
        const uint4 uh = *reinterpret_cast<const uint4*>(wm_hi + static_cast<long long>(n) * C + h * D + v);
        const uint4 ul = *reinterpret_cast<const uint4*>(wm_lo + static_cast<long long>(n) * C + h * D + v);
        const __half2* ph = reinterpret_cast<const __half2*>(&uh);
        const __half2* pl = reinterpret_cast<const __half2*>(&ul);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float2 x = __half22float2(ph[q]), y = __half22float2(pl[q]);
            const float w0 = x.x + y.x, w1 = x.y + y.y;
#pragma unroll
            for (int d = 0; d < 4; ++d) a[d] = fmaf(kv[d][v + 2 * q + 1], w1, fmaf(kv[d][v + 2 * q], w0, a[d]));
        }
    }
    uint2 uh2, ul2;
    split_f16x2(a[0], a[1], uh2.x, ul2.x);
    split_f16x2(a[2], a[3], uh2.y, ul2.y);
    const long long o = (static_cast<long long>(seg) * C + n) * C + h * D + ds * 4;
    *reinterpret_cast<uint2*>(g_hi + o) = uh2;
    *reinterpret_cast<uint2*>(g_lo + o) = ul2;
}

// --------------------------------------------------------------------------------------------------------
// merge per-column-tile softmax partials (log2 domain) into lse[i] = max + log2(sum 2^(. - max))
static __global__ void stats_merge_kernel(const float2* __restrict__ part, int T, int M, float* __restrict__ lse) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    float m = -INFINITY;
    for (int t = 0; t < T; ++t) m = fmaxf(m, part[static_cast<long long>(t) * M + i].x);
    float s = 0.f;
    for (int t = 0; t < T; ++t) {
        const float2 p = part[static_cast<long long>(t) * M + i];
        s += p.y * exp2f(p.x - m);
    }
    lse[i] = m + log2f(s);
}

// Mutual-nearest-neighbour selection + ordered compaction (CoarseMatching.get_coarse_match,
// third_party/LoFTR/src/loftr/utils/coarse_matching.py:172-193).  One CTA of 1024 threads walks the rows in order.
// mask_border quirk: only the LEADING `border` rows/cols of each grid axis are removed (:8-22).
static __global__ void __launch_bounds__(1024) match_select_kernel(const unsigned long long* __restrict__ row_best,
                                                            const unsigned long long* __restrict__ col_best, int L, int w0c, int w1c,
                                                            int border, int capacity, int* __restrict__ i_ids, int* __restrict__ j_ids,
                                                            float* __restrict__ mconf, int* __restrict__ count) {
    __shared__ int warp_sums[32];
    __shared__ int base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i0 = 0; i0 < L; i0 += 1024) {
        const int i = i0 + threadIdx.x;
        int flag = 0, j = 0;
        float conf = 0.f;
        if (i < L) {
            const unsigned long long rb = row_best[i];
            if (rb != 0ull) {
                conf = __uint_as_float(static_cast<unsigned int>(rb >> 32));
                j = 0x7fffffff - static_cast<int>(rb & 0xffffffffu);
                const unsigned long long cb = col_best[j];
                const bool mutual = static_cast<unsigned int>(cb >> 32) == static_cast<unsigned int>(rb >> 32);
                const bool inb = (i / w0c >= border) && (i % w0c >= border) && (j / w1c >= border) && (j % w1c >= border);
                flag = (mutual && inb && conf != 0.f) ? 1 : 0;
            }
        }
        const unsigned int bal = __ballot_sync(0xffffffffu, flag);
        const int wpre = __popc(bal & ((1u << lane) - 1));
        if (lane == 0) warp_sums[warp] = __popc(bal);
        __syncthreads();
        int woff = 0;
        for (int w = 0; w < warp; ++w) woff += warp_sums[w];
        const int pos = base + woff + wpre;
        if (flag && pos < capacity) {
            i_ids[pos] = i;
            j_ids[pos] = j;
            mconf[pos] = conf;
        }
        __syncthreads();
        if (threadIdx.x == 1023) base = pos + flag;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}

}  // namespace dfsfm
