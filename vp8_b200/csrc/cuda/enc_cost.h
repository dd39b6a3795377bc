/*
 * enc_cost.h -- the motion search's cost, shared by the inter-frame encoder kernel (enc_kernels.cu) and its CPU
 * restatement (oracle_inter/enc_inter_oracle.c), so that both pick the same vectors.  Plain C.
 *
 * cost(v) = SAD(source, prediction with v) + lambda * R(v)
 *   R(v)    = bits of the vector relative to the zero vector: per component of magnitude a quarter pels,
 *             0 for a = 0, else 2 * bitlength(a) + 1 (a rough size of its coding as a NEW delta from zero).
 *             Neighbours' vectors are not an input, so every macroblock searches on its own.
 *   lambda  = SAD units per bit, 1 + (y1_ac >> 4), y1_ac = the luma AC quantiser factor of the frame.
 * Largest cost: 16 * 16 * 255 + (1 + 284 / 16) * 2 * 23 < 2^17.
 */
#ifndef VP8R_ENC_COST_H_
#define VP8R_ENC_COST_H_

#if defined(__CUDACC__)
#define VP8R_ENC_FN static __host__ __device__ __forceinline__
#else
#define VP8R_ENC_FN static inline
#endif

VP8R_ENC_FN int vp8r_enc_lambda(int y1_ac) { return 1 + (y1_ac >> 4); }

VP8R_ENC_FN int vp8r_enc_mv_comp_bits(int q) {
  int a = q < 0 ? -q : q, n = 0;
  while (a >> n) ++n;
  return a ? 2 * n + 1 : 0;
}

/* v = (row, col) in quarter pels */
VP8R_ENC_FN int vp8r_enc_mv_bits(int qr, int qc) { return vp8r_enc_mv_comp_bits(qr) + vp8r_enc_mv_comp_bits(qc); }

/* The eight neighbours of a sub-pel refinement step, in scan order (the lowest index wins a tie; the centre, index 0,
 * wins over all of them): step * (dr, dc) with (dr, dc) = (-1,-1) (-1,0) (-1,1) (0,-1) (0,1) (1,-1) (1,0) (1,1). */
VP8R_ENC_FN int vp8r_enc_ring_dr(int k) { return k < 3 ? -1 : (k < 5 ? 0 : 1); }
VP8R_ENC_FN int vp8r_enc_ring_dc(int k) { return k < 3 ? k - 1 : (k < 5 ? (k == 3 ? -1 : 1) : k - 6); }

#endif /* VP8R_ENC_COST_H_ */
