// K6c: the cluster-resident recurrence kernels (rnn_cluster.cu) behind ercg_lstm_* / ercg_gru_* for Hd in
// [RNN_CLUSTER_MIN_HD, RNN_CLUSTER_MAX_HD].  Same arguments and saved-tensor layouts as K6 (lstm.cu) and K6b (gru.cu).
#pragma once
#include "common.cuh"

namespace ercg {

constexpr int RNN_CLUSTER_MIN_HD = 101, RNN_CLUSTER_MAX_HD = 384;

int lstm_cluster_fwd(const float* gx, long long ldgx, const float* whh, const int* node_off, int B, int Hd, float* out,
                     long long ldo, float* gates, float* cells, float* hprev, cudaStream_t st);
int lstm_cluster_bwd(const float* dout, long long ldo, const float* gates, const float* cells, const float* whh,
                     const int* node_off, int B, int Hd, float* dgx, long long lddgx, cudaStream_t st);
int gru_cluster_fwd(const float* gx, long long ldgx, const float* whh, const float* bhh, const int* node_off, int B, int Hd,
                    float* out, long long ldo, float* gates, float* hprev, cudaStream_t st);
int gru_cluster_bwd(const float* dout, long long ldo, const float* gates, const float* hprev, const float* whh,
                    const int* node_off, int B, int Hd, float* dgx, long long lddgx, float* dgh, long long lddgh,
                    cudaStream_t st);

}  // namespace ercg
