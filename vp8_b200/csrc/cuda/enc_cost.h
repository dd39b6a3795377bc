/*
 * enc_cost.h -- the motion search's cost and the intra / inter decision's bias, shared by the inter-frame encoder kernel (enc_kernels.cu) and its CPU
 * restatement (oracle_inter/enc_inter_oracle.c), so that both pick the same vectors and the same intra macroblocks.  Plain C.
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

/* Intra macroblocks of inter frames (VP8R_ENC_INTRA_MBS): a macroblock is coded intra iff
 *   intra_err + vp8r_enc_intra_bias(y1_ac) < inter_err
 * with both errors luma sums of squared prediction errors over the 256 pixels (the intra one of the best 16x16 mode, or
 * of the B_PRED trial when that is strictly better).  bias = y1_ac^2, about three times the
 * quantisation noise a macroblock carries in either choice (256 pixels * (y1_ac / 8)^2 / 12): intra must win by more than
 * that noise.  Measured with the oracle: an unchanged picture, whose inter error is the noise itself, keeps every
 * macroblock inter at q 20, 60 and 127 (with no bias, 6 of 99 went intra at q 127), but at q 0, where the bias is 16,
 * 15 of 8160 macroblocks of a 1920x1080 static scene go intra; a scene cut goes intra almost everywhere with B_PRED
 * (every macroblock of a 176x144 cut at q 20 and 60, 95 % at q 127).
 * Non-negative, non-decreasing in y1_ac; at most 284^2 for y1_ac <= 284, so intra_err + bias < 256 * 255^2 + 284^2
 * fits 32 bits. */
VP8R_ENC_FN int vp8r_enc_intra_bias(int y1_ac) { return y1_ac * y1_ac; }

#endif /* VP8R_ENC_COST_H_ */
