/* liblasr -- CTC Viterbi forced alignment (the same library and conventions as lasr.h: device pointers, `stream` as void*,
 * no host synchronisation, CUDA-graph capturable, 0 or a negative LASR_ERR_* with lasr_last_error()).
 *
 * The reference ships no aligner; this is the project's definition, taken over the CTC head's log-probabilities
 * (nets/ctc.py:25-26: log_softmax(ctc_lo(x)), no dropout).  For utterance b with T = frames[b] frames and the label sequence
 * y = targets[b, :L], L = tgt_len[b], the extended labels are z[2k] = blank, z[2k+1] = y[k] (S = 2L+1 states) and
 *     e[t,s]     = float(logits[b*Tmax + t, z[s]]) - lse[b*Tmax + t]                  one fp32 subtraction
 *     delta[0,s] = e[0,s] for s in {0, 1}, -inf otherwise
 *     delta[t,s] = max(delta[t-1,s], delta[t-1,s-1], delta[t-1,s-2]) + e[t,s]        one fp32 add
 * where s-2 is a predecessor only when s is odd, s >= 3 and z[s] != z[s-2].
 *   Ties: the higher predecessor index wins (stay on s, then s-1, then s-2).  End state: the better of S-1 and S-2; a tie goes to
 *   S-1 (a trailing blank).  L = 0 gives the all-blank path.  max is exact and each step is one rounded add, so a float32
 *   restatement of these lines reproduces every output bit for bit.
 * Outputs (device):
 *   state      (B, Tmax) int32: the state s of the best path on each frame; -1 on frames t >= T
 *   frame_logp (B, Tmax) fp32 : e[t, state[t]]; -inf on frames t >= T
 *   score      (B,)      fp32 : the optimum delta
 *   spans      (B, lmax, 2) int32: first and last frame of label k (the frames of a label form one run); -1 for k >= L
 * An utterance whose frames cannot hold its transcript (T < L + the number of adjacent repeated labels), or whose optimum is
 * -inf for another reason (T = 0, a label outside [0, V) whose emission is -inf), is not an error: its score is -inf and all
 * its state / spans entries are -1 and its frame_logp entries -inf.
 * Inputs: logits (B*Tmax, >= V) fp32 | bf16 (dtype), row stride ld >= V, utterance b at rows [b*Tmax, b*Tmax + frames[b]);
 *   lse (B*Tmax,) fp32 row log-sum-exp (lasr_logsoftmax_topk's `lse`); targets (B, lmax) int64 (entries past tgt_len[b]
 *   ignored, -1 by convention); tgt_len, frames (B,) int64, clamped to [0, lmax] / [0, Tmax]; 0 <= blank < V.
 * Limits: lmax <= 16383 (S <= 32767) and Tmax <= 16384; larger sizes return LASR_ERR_BAD_ARG with a message naming the bound.
 * Workspace: lasr_ctc_forced_align_workspace(B, Tmax, lmax) bytes of 2-bit back-pointers (0 for arguments outside the limits):
 *   B * Tmax * NT * 8 with NT = clamp(roundup32(ceil(S/8)), 32, 1024) threads per utterance for S = 2 lmax + 1, about
 *   Tmax * S / 4 bytes per utterance for long transcripts (134 MB at Tmax = 16384, lmax = 16383).
 * One launch for the whole batch: one CTA per utterance (its shape chosen from lmax), lattice row in shared memory.
 */
#ifndef LASR_ALIGN_H
#define LASR_ALIGN_H

#include "lasr.h"

#ifdef __cplusplus
extern "C" {
#endif

size_t lasr_ctc_forced_align_workspace(int B, int Tmax, int lmax);
int lasr_ctc_forced_align(const void* logits, int dtype, int64_t ld, const float* lse, const int64_t* targets, const int64_t* tgt_len,
                          const int64_t* frames, int B, int Tmax, int lmax, int V, int blank, int32_t* state, float* frame_logp,
                          float* score, int32_t* spans, void* workspace, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LASR_ALIGN_H */
