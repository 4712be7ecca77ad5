// Shared between the beam search (beam.cu) and the caption sampler (sample.cu): the workspace layout and the host-side pieces
// of both decoders' generation loops — the once-per-call prologue, the per-step decoder computation on the live rows (ending in
// w.logits), and the start / compaction / reorder launches of the slot state machine.
#pragma once
#include "common.cuh"

struct BeamWs {
    float *att_enc, *mean, *h0, *c0, *h, *c, *h_tmp, *c_tmp, *w_cat, *b_cat, *emb_x, *z, *gated, *gates_pre,
          *gates_act_unused, *logits, *alpha_steps, *score, *best_score, *embg;
    int *img_index, *prev_word, *k_live, *src, *parent, *word, *best_step, *best_parent;
    int *slot_img, *slot_img_tmp, *k_live_tmp, *new_slot, *n_live, *word_tmp;   // n_live[0] = live slots, [1] = live rows
    int* ring_ticket;                                                           // one slot-ticket counter per step (attention ring kernel)
    int *row_off[2];                                                            // slot -> first state row (ping-pong per step)
    float* score_tmp;
    long long* tok64;
    // ICD_PREC_FP32X3: 3-term bf16 splits (gemm_tc.cu) of the weights (once per call) and of the step activations
    void *x3_We, *x3_Wcat, *x3_WihE, *x3_WihC, *x3_Wh, *x3_Wc, *x3_Wfc, *x3_act;
    float* x3_splitk; long long x3_splitk_floats;
    // baseline decoder only (carve_base): fp32 copy of an fp64 embedding table, split of W_hh
    float* emb32;
    void* x3_Whh;
    // sampler only (history == false): per-row sample index, moved with the row by beam_reorder_kernel; NULL in the beam search
    int *tag, *tag_tmp;
};

// history: the beam search's per-step parent / word pointers and alpha frames (S x rows each).  Without it (the sampler) the
// alpha buffer holds one step, there are no parent / word arrays, and the per-row tag arrays are carved instead.
size_t carve(const icd_beam_desc_t* d, BeamWs* w, char* base, bool history = true);
size_t carve_base(const icd_base_beam_desc_t* d, BeamWs* w, char* base, bool history = true);

// Attention decoder.  Prologue: weight concatenation and splits, whole-vocabulary embg, att_enc, the initial state h0 / c0.
// *use_embg tells the step whether the embedding contraction became a row gather.  Step: logits of the live rows into w.logits,
// the attention weights of the step into alpha_s (rows of P).
int beam_att_prologue(const icd_beam_desc_t* d, BeamWs& w, bool* use_embg, cudaStream_t s);
int beam_att_step(const icd_beam_desc_t* d, BeamWs& w, int step, bool use_embg, const int* row_off, float* alpha_s, cudaStream_t s);
// Baseline decoder.  Prologue: weight splits, embg, the image step (h0 / c0).  Step: h W_hh^T, the fused cell, the vocabulary layer.
int beam_base_prologue(const icd_base_beam_desc_t* d, BeamWs& w, cudaStream_t s);
int beam_base_step(const icd_base_beam_desc_t* d, BeamWs& w, cudaStream_t s);
// One live row per image (state h0 / c0, previous word start_id, score 0), one slot per image.
int beam_launch_init(int n_img, int k, int D, int start_id, BeamWs& w, cudaStream_t s);
// After a selection kernel filled the *_tmp arrays: compact the slots, move the surviving rows (and w.tag_tmp -> w.tag if set).
int beam_launch_advance(int n_img, int k, int D, BeamWs& w, const int* row_off, int* row_off_next, cudaStream_t s);
