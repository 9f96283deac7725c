// The seam between the LSTM forward (lstm.cu) and its training backward (lstm_train.cu): the engine handle, the tape
// layout, the backward's graph cache and entry points, and the kernel both use to shift lengths by one position.
#pragma once

#include "common.cuh"

namespace avvad {
struct BpttGraphCache;  // cached CUDA graphs of the backward recurrence (lstm_train.cu)
BpttGraphCache* bptt_cache_create();
void bptt_cache_destroy(BpttGraphCache* c);
}  // namespace avvad

struct avvad_lstm {
  int layers, input_size, H, y_dim;
  int64_t ld0;               // padded layer-0 input width
  __nv_bfloat16* w_ih[8];    // [4H][ld_l]
  __nv_bfloat16* w_hh[8];    // [4H][H]
  float* bias[8];            // [4H] gate-interleaved, b_ih + b_hh
  float* head_w32;           // [y_dim][H]
  __nv_bfloat16* head_w16;   // [y_dim][H]
  float* head_b;             // [y_dim]
  bool set[8];
  bool head_set;
  avvad::BpttGraphCache* bptt;
  // layer overlap (lstm_forward_impl): layer 1 follows layer 0 one chunk of time steps behind on a side stream
  cudaStream_t side = nullptr;
  int side_device = -1;
  cudaEvent_t ev_chunk[32] = {};
  cudaEvent_t ev_done = nullptr;
};

namespace avvad {
// One layer of the training tape (avvad_lstm_tape_layout): gates bf16 [B][T][4H] (gate-interleaved, element 4u+g),
// c f32 [B][T][H], hseq bf16 [B][T][H]
struct TapeView {
  __nv_bfloat16* gates;
  float* c;
  __nv_bfloat16* hseq;
};
TapeView tape_layer(void* tape, int l, int H, int64_t B, int64_t T);

// A stateful call runs its steps at positions 1..T of sequences whose position 0 holds the state: out[b] = lengths[b] + 1
__global__ void shift_lengths_kernel(const int32_t* __restrict__ lengths, int B, int32_t* __restrict__ out);

// BPTT over a tape of T positions (avvad_lstm_backward); `bs` is null there and is set by the stateful backward
struct BpttState;
size_t lstm_backward_workspace(const avvad_lstm* h, int64_t B, int64_t T);
int lstm_backward_impl(const avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T, void* tape,
                       const float* dlogits, void* workspace, size_t workspace_bytes, float* const* dW_ih,
                       float* const* dW_hh, float* const* db, float* dW_head, float* db_head, float* dx, cudaStream_t st,
                       const BpttState* bs);
// BPTT over a stateful tape of T + 1 positions (avvad_lstm_backward_state)
size_t lstm_backward_state_workspace(const avvad_lstm* h, int64_t B, int64_t T);
int lstm_backward_state_impl(const avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                             void* tape, const float* dlogits, const float* dh_out, const float* dc_out, float* dh_in,
                             float* dc_in, void* workspace, size_t workspace_bytes, float* const* dW_ih,
                             float* const* dW_hh, float* const* db, float* dW_head, float* db_head, float* dx,
                             cudaStream_t st);
}  // namespace avvad
