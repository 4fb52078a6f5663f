// feat_attn_core.cuh — attention between the T feature tokens of ONE table row for ONE head (layer.py:332-339),
// on mma.sync m16n8k16 from a shared-memory block that holds the row's q / k / v as bf16 token rows.
// Shared by the stand-alone feature attention kernel (kernels_f32.cu, reads a qkv block from global memory) and by
// the fused QKV-projection + feature-attention kernel (kernels_featfused.cu, reads what its own GEMM left there).
#pragma once
#include "common.cuh"

namespace mmpfn {

__device__ __forceinline__ void fa_ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void fa_ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
template <int FMT>
__device__ __forceinline__ void fa_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (FMT == FMT_F16)
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  else
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// One warp: queries mt*16 .. mt*16+15 of the row against its T keys.
//   sbase      shared address of the row's first token; token rows are row_bytes apart (16-byte multiple whose
//              residue mod 128 is 16: conflict-free ldmatrix)
//   q_off / k_off / v_off   byte offsets of this head's 32-wide q / k / v block inside a token row
//   n_kt       16-key tiles present (T <= 16 n_kt <= 16 KT); token rows T .. 16 n_kt - 1 must hold FINITE values
//              (their keys are masked, but 0 x NaN in P V would still poison the output)
// FMT: the 16-bit format of q / k / v, P and the output (FMT_BF16 or FMT_F16).
// The normalised output (16-bit) overwrites the head's q block of the query rows < T: 16 tokens x 64 B that only this
// warp reads and holds in registers since its first ldmatrix.
template <int KT, int FMT>
__device__ __forceinline__ void feat_attn_item(uint32_t sbase, int row_bytes, int q_off, int k_off, int v_off, int T,
                                               int n_kt, int mt, int lane) {
  const float c2 = 0.17677669529663687f * 1.4426950408889634f;   // log2(e)/sqrt(d)
  // Q fragments: 16 queries x 32 d = 2 k-steps
  uint32_t qa[2][4];
#pragma unroll
  for (int ks = 0; ks < 2; ++ks)
    fa_ldsm_x4(qa[ks], sbase + (mt * 16 + (lane & 15)) * row_bytes + q_off + (ks * 16 + (lane >> 4) * 8) * 2);
  // S = Q K^T
  float sacc[2 * KT][4];
#pragma unroll
  for (int nt = 0; nt < 2 * KT; ++nt) { sacc[nt][0] = sacc[nt][1] = sacc[nt][2] = sacc[nt][3] = 0.f; }
#pragma unroll
  for (int kt = 0; kt < KT; ++kt) {
    if (kt < n_kt) {
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        uint32_t kb[4];
        const int mi = lane >> 3;
        fa_ldsm_x4(kb, sbase + (kt * 16 + (mi >> 1) * 8 + (lane & 7)) * row_bytes + k_off + (ks * 16 + (mi & 1) * 8) * 2);
        fa_mma<FMT>(sacc[2 * kt], qa[ks], kb[0], kb[1]);
        if (kt * 16 + 8 < T) fa_mma<FMT>(sacc[2 * kt + 1], qa[ks], kb[2], kb[3]);   // (an 8-key tile past T is masked anyway)
      }
    }
  }
  // softmax over the T real keys; thread holds rows (lane/4) and (lane/4 + 8), key columns (lane%4)*2 + {0,1}
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < 2 * KT; ++nt) {
    if (nt < 2 * n_kt) {
      const int key = nt * 8 + (lane & 3) * 2;
      if (key >= T) { sacc[nt][0] = -INFINITY; sacc[nt][2] = -INFINITY; }
      if (key + 1 >= T) { sacc[nt][1] = -INFINITY; sacc[nt][3] = -INFINITY; }
      mx0 = fmaxf(mx0, fmaxf(sacc[nt][0], sacc[nt][1]));
      mx1 = fmaxf(mx1, fmaxf(sacc[nt][2], sacc[nt][3]));
    }
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  const float mc0 = mx0 * c2, mc1 = mx1 * c2;
  float l0 = 0.f, l1 = 0.f;
  float oacc[4][4];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) { oacc[nt][0] = oacc[nt][1] = oacc[nt][2] = oacc[nt][3] = 0.f; }
  // P of one 16-key tile as the A fragment of P V (16-bit), row sums on the side
  auto probs = [&](int kt, uint32_t (&pa)[4]) {
    const float p00 = fast_exp2f(fmaf(sacc[2 * kt][0], c2, -mc0)), p01 = fast_exp2f(fmaf(sacc[2 * kt][1], c2, -mc0));
    const float p10 = fast_exp2f(fmaf(sacc[2 * kt][2], c2, -mc1)), p11 = fast_exp2f(fmaf(sacc[2 * kt][3], c2, -mc1));
    const float q00 = fast_exp2f(fmaf(sacc[2 * kt + 1][0], c2, -mc0)), q01 = fast_exp2f(fmaf(sacc[2 * kt + 1][1], c2, -mc0));
    const float q10 = fast_exp2f(fmaf(sacc[2 * kt + 1][2], c2, -mc1)), q11 = fast_exp2f(fmaf(sacc[2 * kt + 1][3], c2, -mc1));
    l0 += (p00 + p01) + (q00 + q01);
    l1 += (p10 + p11) + (q10 + q11);
    pa[0] = pack16x2<FMT>(p00, p01); pa[1] = pack16x2<FMT>(p10, p11);
    pa[2] = pack16x2<FMT>(q00, q01); pa[3] = pack16x2<FMT>(q10, q11);
  };
#pragma unroll
  for (int kt = 0; kt < KT; ++kt) {
    if (kt < n_kt) {
      uint32_t pa[4];
      probs(kt, pa);
#pragma unroll
      for (int np = 0; np < 2; ++np) {
        uint32_t vb[4];
        const int mi = lane >> 3;
        fa_ldsm_x4_t(vb, sbase + (kt * 16 + (mi & 1) * 8 + (lane & 7)) * row_bytes + v_off + (np * 16 + (mi >> 1) * 8) * 2);
        fa_mma<FMT>(oacc[2 * np], pa, vb[0], vb[1]);
        fa_mma<FMT>(oacc[2 * np + 1], pa, vb[2], vb[3]);
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
  const int q0 = mt * 16 + (lane >> 2), q1 = q0 + 8;
  const uint32_t so0 = sbase + q0 * row_bytes + q_off + (lane & 3) * 4;
  const uint32_t so1 = sbase + q1 * row_bytes + q_off + (lane & 3) * 4;
  __syncwarp();
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    if (q0 < T)
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(so0 + nt * 16), "r"(pack16x2<FMT>(oacc[nt][0] * i0, oacc[nt][1] * i0)) : "memory");
    if (q1 < T)
      asm volatile("st.shared.b32 [%0], %1;" ::"r"(so1 + nt * 16), "r"(pack16x2<FMT>(oacc[nt][2] * i1, oacc[nt][3] * i1)) : "memory");
  }
}

}  // namespace mmpfn
