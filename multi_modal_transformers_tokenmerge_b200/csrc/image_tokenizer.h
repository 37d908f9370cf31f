// Internal interface of the image front end (image_tokenizer.cu) for the pixels-to-actions call in stack.cu
// (tome_policy_predict): the front end writing its tokens straight into the rows of an assembled [B, T0, C] sequence, and
// the kernel that fills the sequence's other rows.  Not part of the C ABI.
#pragma once
#include "host_util.h"

namespace tome {

// Image token k = n * n_patches + p of every batch row goes to sequence row row0[i] + (k - k0[i]) for the run i with
// k0[i] <= k < k0[i + 1] (k0[n_runs] = N * n_patches).  A grammar's image sets are contiguous runs of rows, so a handful of
// runs describes the placement; the runs travel to the kernel by value.
constexpr int IT_MAX_ROW_RUNS = 32;
struct ItPlacement {
  int n_runs;
  int seq_tokens;   // T0
  int n_images;     // N
  int k0[IT_MAX_ROW_RUNS + 1];
  int row0[IT_MAX_ROW_RUNS];
};

// The non-image rows: set s copies src[s] (bf16 [B or 1, n[s], C], batch_stride[s] elements between batch rows, 0 = one
// set for every row) to sequence rows row0[s] .. row0[s] + n[s] - 1.
struct SeqRowSets {
  int n_sets;
  const void* src[TOME_MAX_TOKEN_SETS];
  long long batch_stride[TOME_MAX_TOKEN_SETS];
  int n[TOME_MAX_TOKEN_SETS];
  int row0[TOME_MAX_TOKEN_SETS];
};

// tome_image_tokenizer_fwd with the final stage writing bf16 token (b, n, p) to seq[b, row(n * n_patches + p), :] (desc->out_dtype
// must be TOME_BF16).  Same validation and the same bits as the dense output.
int image_tokenizer_fwd_placed(const tome_image_tokenizer_desc_t* d, const void* image, const float* pf, const void* pb,
                               const int32_t* row_tokens, const int32_t* col_tokens, const ItPlacement& place, void* seq,
                               void* workspace, size_t workspace_bytes, cudaStream_t stream);

// One launch: every set of `sets` into the bf16 sequence [batch, seq_tokens, channels] (bit copies).
int fill_sequence_rows(const SeqRowSets& sets, int batch, int seq_tokens, int channels, void* seq, cudaStream_t stream);

}  // namespace tome
