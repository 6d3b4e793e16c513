// Replica-batched MLP forward / backward programs built from the grouped GEMM (gemm.cu).
#pragma once
#include "common.cuh"

// A grouped row-major matrix view: element (g, i, j) at ptr + (g / gdiv) * gs + i * ld + j.
struct MatView {
  const float* ptr;
  int64_t gs;
  int gdiv;
  int ld;
};

struct MlpActs {  // outputs of the hidden layers ([G, n, dims[l+1]] contiguous), kept for the backward pass
  float* hid[IL_MAX_LAYERS];
  // ReLU sign bits of the same outputs ([G, n, dims[l+1] / 32] words): what a backward pass needs of an activation that only serves as the derivative mask.
  // Carved for widths that are multiples of 32; bits_valid[l] is set by mlp_forward when the kernel that produced hid[l] also wrote the words.
  uint32_t* bits[IL_MAX_LAYERS];
  bool bits_valid[IL_MAX_LAYERS];
};
enum { MLP_KEEP_NONE = 0, MLP_KEEP_ALL = 1, MLP_KEEP_MASKS = 2 };  // what the forward pass keeps: nothing / activations for a full backward / only what an input-gradient pass needs

// Bytes for the hidden activations of G nets on n rows (il_align_up'ed per buffer).
int64_t mlp_acts_bytes(const il_mlp* m, int G, int n);
// Carves hidden-activation buffers out of `ws`; returns the advanced pointer.
char* mlp_acts_carve(const il_mlp* m, int G, int n, char* ws, MlpActs* acts);

// Forward of G nets: out[g] ([n, dims[L]], row stride ld_out, group stride out_gs) = net_g(X[g]).
// keep == MLP_KEEP_NONE: the hidden activations are not needed afterwards (no backward pass follows), which lets the fused head epilogue skip
// writing the last hidden layer. MLP_KEEP_MASKS: only mlp_backward(grads = nullptr, dX) follows — the last hidden layer is kept as sign bits only
// when the kernels support it. (bool arguments convert: false = NONE, true = ALL.)
int mlp_forward(il_handle* h, const il_mlp* m, int G, int n, MatView X, MlpActs& acts, float* out, int64_t out_gs, int ld_out,
                cudaStream_t stream, int keep = MLP_KEEP_ALL);

// Backward of G nets from dOut (gradient at the linear head), using the saved hidden outputs.
//  grads != nullptr : parameter gradients written in the flat parameter layout (net stride grad_stride).
//  dX    != nullptr : gradient w.r.t. input columns [dx_col0, dx_col0 + dx_cols) written to dX (ld_dx, group stride dx_gs).
//  tmpA / tmpB      : two scratch buffers of G * n * max_hidden floats (ping-pong for the layer gradients).
int mlp_backward(il_handle* h, const il_mlp* m, int G, int n, MatView X, const MlpActs& acts, MatView dOut, float* grads, int64_t grad_stride,
                 float* dX, int64_t dx_gs, int ld_dx, int dx_col0, int dx_cols, float* tmpA, float* tmpB, cudaStream_t stream);

// Whole-MLP forward in one kernel for n <= 32 rows per net (rollout / evaluation rows). tanh_first = A > 0 writes only
// tanh of the first A outputs ([G, n, A]): the greedy action of a SoftActor (models.py:101-102).
int mlp_small_forward(il_handle* h, const il_mlp* m, int G, int n, MatView X, float* out, cudaStream_t stream, int tanh_first = 0);
int mlp_max_hidden(const il_mlp* m);
int mlp_validate(const il_mlp* m, const char* what);

// ---- tanh-Gaussian head (mlp.cu) ---------------------------------------------------------------------------
struct HeadFwdArgs {
  const float* head;        // [rows, 2A] raw actor output (mean | log-std)
  const float* eps;         // [rows, A] or nullptr
  const float* given;       // [rows, A] or nullptr (log-prob of a given action, atanh path)
  float* action;            // nullable; element (r, i, j) at action + r * action_rs + i * ld_action + j
  int64_t action_rs;
  int ld_action;
  const float* zero_mask;   // nullable [rows]: action *= (1 - zero_mask[row])   (training.py:23)
  int64_t zero_mask_rs;     // replica stride of zero_mask (row i of replica r at zero_mask + r*rs + i*zero_mask_ld)
  int zero_mask_ld;
  float* log_prob;          // nullable [rows]
  float* mean;              // nullable [rows, A]
  float* log_std;           // nullable [rows, A]
  const float* copy_src;    // nullable: copy `copy_cols` floats of row (r, i) from copy_src + r*copy_rs + i*copy_ld to action row start - copy_cols
  int64_t copy_rs;
  int copy_ld, copy_cols;
  int R, n, A;
};
int launch_actor_head(il_handle* h, const HeadFwdArgs& a, cudaStream_t stream);

// polyak_target != nullptr: also applies update_target_network (models.py:79-81) with the freshly stepped parameters
// polyak_r (nullable [R]): per-replica polyak factor, replica r = floats [r * opt->replica_floats, (r + 1) * opt->replica_floats)
int launch_adam(il_handle* h, float* params, const float* grads, const il_adam* opt, int64_t n, cudaStream_t stream, float* polyak_target = nullptr, float polyak_factor = 0.f,
                const float* polyak_r = nullptr);
int launch_tick(il_handle* h, int64_t* s0, int64_t* s1, int64_t* s2, cudaStream_t stream);
