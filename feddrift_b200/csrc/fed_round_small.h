// Argument block of the fused persistent FL-round kernel (fed_round_small.cu).
#pragma once
#include <cuda_runtime.h>

namespace fdb {

constexpr int kMaxPeers = 8;

struct RoundParams {
    // data (device-resident for the whole experiment)
    const float* X;      // [T1, C, S, IN]
    const int* Y;        // [T1, C, S]
    const int* nsamp;    // [T1, C]
    // plan
    float* W;                  // [t_cur+1, M, C]   (rewritten in place by IFCA re-clustering)
    const int* train_index;    // [M, C, Lmax] flat (t'*S + s) sample ids   (sample_mode == 2)
    const int* train_count;    // [M, C]
    const float* feat_mask;    // [M, IN] or nullptr (training inputs only)
    const int* eval_train_model;  // [C] or nullptr (-1 → argmax_m W[t, m, c])
    const int* eval_test_model;   // [C] or nullptr
    const float* ens_w;        // [C, M] or nullptr
    // model / optimizer state
    float* theta;        // [M, theta_stride]
    float* opt_m;        // [C, M, P]  (row s·M + m: worker slot s, see participants)
    float* opt_v;
    float* opt_vmax;
    int* opt_step;       // [C, M]
    float* client_out;   // optional [C, M, P] export of the local models of the LAST round (nullptr = off); slot-indexed
    // partial participation: row (round0 + r) % part_rows of this table lists the K clients that train in round r;
    // optimizer state and client_out rows then belong to worker slot s (the s-th listed client), not to client s.
    // nullptr = every client trains every round (slot == client).
    const int* participants;   // [part_rows, K] distinct client ids, or nullptr
    int K, part_rows;
    const float* lr_ptr; // optional device scalar overriding lr
    // outputs
    float* metrics;      // [rounds, C, 4]
    long long* timers;   // optional [rounds, 4] globaltimer ns stamps of CTA 0 (train end, agg end, eval end, -)
    int* counters;       // optional device counters {round_in_step, global_epoch}: read at start, advanced at exit
    // scalars
    float lr, wd, beta1, beta2, eps;
    int T1, C, S, M, Lmax, theta_stride;
    int batch_size, epochs, t_cur, rounds, round0;
    unsigned seed;
    int use_adam;       // 1 = Adam(amsgrad, L2 wd), 0 = SGD
    int sample_mode;    // 0 pool, 1 time-weighted, 2 explicit index lists
    int n_mode;         // 0 Σ W·nb, 1 Σ W·nsamp       (pool mode only)
    int recluster_hard; // IFCA: argmax re-clustering after every aggregation
    int ens_mode;       // 0 none, 1 weighted hard vote, 2 weighted soft vote (test metric)
    int skip_aggregate; // 1 = train + export only (CFL inspects raw updates)
    int warps_per_pair; // 1, 2 or 4 warps cooperate on one (client, model) pair
    // multi-GPU (clients sharded c % world == rank); world == 1 → everything local
    int world, rank;
    float* inbox[kMaxPeers];     // inbox[g]: this rank's view of peer g's symmetric inbox: LL words {value, epoch} [2, world, M*P] x 8 B
    float* metrics_peer[kMaxPeers];  // every rank's (symmetric) metrics STAGING area: LL words {corr, epoch, loss, epoch} [rounds, C, 2] x 16 B
    unsigned flag_base;          // monotonically increasing epoch base (per launch)
    long long spin_timeout_ns;   // bail out instead of hanging the GPU if a peer never arrives
    int* error_flag;             // set to nonzero on timeout
    // fused host I/O (single-GPU end-to-end round): the kernel itself performs the host→device copy of the round's inputs
    // from PINNED host memory (UVA pointers; 16-byte system-scope loads over PCIe) into the X / Y arenas before round 0,
    // and mirrors every metric row into a pinned host buffer — the whole round is ONE graph node, no memcpy nodes.
    const float* host_x;         // pinned [host_steps, C, S, IN] or nullptr
    const int* host_y;           // pinned [host_steps, C, S]
    float* host_metrics;         // pinned [rounds, C, 4] or nullptr
    int host_t0, host_steps;     // destination time steps [host_t0, host_t0 + host_steps)
};

struct SmallLaunchInfo {
    int threads, cluster, smem_bytes;
};

// returns 0 on success, -1 if (kind,in,hid,out) is not an instantiated shape
int fed_round_small_launch(int kind, int din, int hid, int dout, const RoundParams& p, int cluster, cudaStream_t stream,
                           SmallLaunchInfo* info);
int fed_round_small_supported(int kind, int din, int hid, int dout);
int fed_round_small_fits(int kind, int din, int hid, int dout, int C, int M, int t_cur);
// cluster size the launcher uses (or -1: shape not instantiated) and its dynamic shared memory in *smem (> 227 KB: no launch)
int fed_round_small_launch_shape(int kind, int din, int hid, int dout, int C, int M, int slots, int cluster,
                                 int warps_per_pair, int* smem);
int mlp_eval_matrix_launch(int kind, int din, int hid, int dout, const float* theta, int theta_stride, int M, const float* X,
                           const int* Y, const int* nsamp, int C, int S, float* correct, float* loss, float* sqerr,
                           cudaStream_t stream);

}  // namespace fdb
