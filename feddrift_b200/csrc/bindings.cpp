// pybind / torch bindings for the feddrift_b200 sm_100a kernels.  All launches go to the current CUDA stream.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include "fed_round_small.h"
#include "kernels.h"

namespace {

using torch::Tensor;

inline cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }
#define CHECK_CUDA_F32(x) TORCH_CHECK((x).is_cuda() && (x).scalar_type() == torch::kFloat32, #x " must be a CUDA float32 tensor")
#define CHECK_CUDA_I32(x) TORCH_CHECK((x).is_cuda() && (x).scalar_type() == torch::kInt32, #x " must be a CUDA int32 tensor")
#define CHECK_OK(code, what) TORCH_CHECK((code) == 0, what, " failed with code ", (code))

template <typename T>
T* opt_ptr(const c10::optional<Tensor>& t) { return (t.has_value() && t->defined()) ? t->data_ptr<T>() : nullptr; }

// ---------------------------------------------------------------------------------- fused small round
// `cfg` carries the scalar fields; tensors are passed explicitly.  Returns (cluster, threads, smem_bytes).
std::vector<int64_t> fed_round_small(
    int64_t kind, int64_t din, int64_t hid, int64_t dout, Tensor X, Tensor Y, Tensor nsamp, Tensor W, Tensor theta, int64_t theta_stride,
    c10::optional<Tensor> opt_m, c10::optional<Tensor> opt_v, c10::optional<Tensor> opt_vmax, Tensor opt_step,
    c10::optional<Tensor> train_index, c10::optional<Tensor> train_count, c10::optional<Tensor> feat_mask,
    c10::optional<Tensor> eval_train_model, c10::optional<Tensor> eval_test_model, c10::optional<Tensor> ens_w,
    c10::optional<Tensor> client_out, c10::optional<Tensor> lr_dev, Tensor metrics, c10::optional<Tensor> timers,
    std::vector<double> fcfg, std::vector<int64_t> icfg, std::vector<int64_t> peer_inbox,
    c10::optional<Tensor> error_flag, c10::optional<Tensor> counters, std::vector<int64_t> peer_metrics, std::vector<int64_t> host_io,
    c10::optional<Tensor> participants) {
    CHECK_CUDA_F32(X); CHECK_CUDA_I32(Y); CHECK_CUDA_I32(nsamp); CHECK_CUDA_F32(W); CHECK_CUDA_F32(theta); CHECK_CUDA_I32(opt_step);
    CHECK_CUDA_F32(metrics);
    TORCH_CHECK(X.is_contiguous() && Y.is_contiguous() && nsamp.is_contiguous() && W.is_contiguous() && metrics.is_contiguous(),
                "fed_round_small: tensors must be contiguous");
    c10::cuda::CUDAGuard guard(X.device());
    fdb::RoundParams p{};
    p.X = X.data_ptr<float>(); p.Y = Y.data_ptr<int>(); p.nsamp = nsamp.data_ptr<int>();
    p.W = W.data_ptr<float>();
    p.train_index = opt_ptr<int>(train_index); p.train_count = opt_ptr<int>(train_count);
    p.feat_mask = opt_ptr<float>(feat_mask);
    p.eval_train_model = opt_ptr<int>(eval_train_model); p.eval_test_model = opt_ptr<int>(eval_test_model);
    p.ens_w = opt_ptr<float>(ens_w);
    p.theta = theta.data_ptr<float>();
    p.opt_m = opt_ptr<float>(opt_m); p.opt_v = opt_ptr<float>(opt_v); p.opt_vmax = opt_ptr<float>(opt_vmax);
    p.opt_step = opt_step.data_ptr<int>();
    p.client_out = opt_ptr<float>(client_out);
    // [rows, K] int32 client ids per round (validated by ops/small_round.py before the launch)
    p.participants = opt_ptr<int>(participants);
    if (p.participants) { p.part_rows = (int)participants->size(0); p.K = (int)participants->size(1); }
    p.lr_ptr = opt_ptr<float>(lr_dev);
    p.metrics = metrics.data_ptr<float>();
    p.timers = (timers.has_value() && timers->defined()) ? reinterpret_cast<long long*>(timers->data_ptr<int64_t>()) : nullptr;
    // fcfg: lr, wd, beta1, beta2, eps
    p.lr = (float)fcfg[0]; p.wd = (float)fcfg[1]; p.beta1 = (float)fcfg[2]; p.beta2 = (float)fcfg[3]; p.eps = (float)fcfg[4];
    // icfg: T1, C, S, M, Lmax, batch, epochs, t_cur, rounds, round0, seed, use_adam, sample_mode, n_mode, recluster, ens_mode,
    //       skip_aggregate, world, rank, flag_base, cluster, spin_timeout_ms
    p.T1 = (int)icfg[0]; p.C = (int)icfg[1]; p.S = (int)icfg[2]; p.M = (int)icfg[3]; p.Lmax = (int)icfg[4];
    p.theta_stride = (int)theta_stride;
    p.batch_size = (int)icfg[5]; p.epochs = (int)icfg[6]; p.t_cur = (int)icfg[7]; p.rounds = (int)icfg[8]; p.round0 = (int)icfg[9];
    p.seed = (unsigned)icfg[10]; p.use_adam = (int)icfg[11]; p.sample_mode = (int)icfg[12]; p.n_mode = (int)icfg[13];
    p.recluster_hard = (int)icfg[14]; p.ens_mode = (int)icfg[15]; p.skip_aggregate = (int)icfg[16];
    p.world = (int)icfg[17]; p.rank = (int)icfg[18]; p.flag_base = (unsigned)icfg[19];
    const int cluster = (int)icfg[20];
    p.spin_timeout_ns = (long long)icfg[21] * 1000000LL;
    p.warps_per_pair = icfg.size() > 22 ? (int)icfg[22] : 1;
    TORCH_CHECK(p.t_cur < 64, "fed_round_small supports t_cur < 64 time steps (use fed_round_small_fits to route)");
    TORCH_CHECK(p.world >= 1 && p.world <= fdb::kMaxPeers, "world must be in [1, 8]");
    if (p.world > 1) {
        TORCH_CHECK((int)peer_inbox.size() == p.world, "need one inbox pointer per rank");
        for (int g = 0; g < p.world; ++g) p.inbox[g] = reinterpret_cast<float*>(peer_inbox[g]);
        TORCH_CHECK(!p.recluster_hard, "per-round IFCA re-clustering is single-GPU only in this build");
    }
    p.error_flag = opt_ptr<int>(error_flag);
    p.counters = opt_ptr<int>(counters);
    for (int g = 0; g < fdb::kMaxPeers; ++g) p.metrics_peer[g] = nullptr;
    if (host_io.size() == 5) {   // {pinned X ptr, pinned Y ptr, pinned metrics ptr, t0, steps}: fused host I/O (see fed_round_small.h)
        p.host_x = reinterpret_cast<const float*>(host_io[0]);
        p.host_y = reinterpret_cast<const int*>(host_io[1]);
        p.host_metrics = reinterpret_cast<float*>(host_io[2]);
        p.host_t0 = (int)host_io[3];
        p.host_steps = (int)host_io[4];
        TORCH_CHECK(p.host_t0 >= 0 && p.host_t0 + p.host_steps <= p.T1, "fed_round_small: host_io time range out of bounds");
    }
    if (p.world > 1 && (int)peer_metrics.size() == p.world)
        for (int g = 0; g < p.world; ++g) p.metrics_peer[g] = reinterpret_cast<float*>(peer_metrics[g]);
    if (p.use_adam) TORCH_CHECK(p.opt_m && p.opt_v && p.opt_vmax, "adam needs optimizer state tensors");
    fdb::SmallLaunchInfo info{};
    const int rc = fdb::fed_round_small_launch((int)kind, (int)din, (int)hid, (int)dout, p, cluster, cur_stream(), &info);
    TORCH_CHECK(rc != -1, "fed_round_small: MLP shape (", kind, ",", din, ",", hid, ",", dout, ") is not instantiated");
    TORCH_CHECK(rc != -2, "fed_round_small: shared-memory footprint exceeds 227 KB for this (clients, models) size");
    CHECK_OK(rc, "fed_round_small launch");
    return {info.cluster, info.threads, info.smem_bytes};
}

bool fed_round_small_fits(int64_t kind, int64_t din, int64_t hid, int64_t dout, int64_t C, int64_t M, int64_t t_cur) {
    return fdb::fed_round_small_fits((int)kind, (int)din, (int)hid, (int)dout, (int)C, (int)M, (int)t_cur) != 0;
}

std::vector<int64_t> fed_round_small_launch_shape(int64_t kind, int64_t din, int64_t hid, int64_t dout, int64_t C, int64_t M,
                                                  int64_t slots, int64_t cluster, int64_t warps_per_pair) {
    int smem = 0;
    const int G = fdb::fed_round_small_launch_shape((int)kind, (int)din, (int)hid, (int)dout, (int)C, (int)M, (int)slots,
                                                    (int)cluster, (int)warps_per_pair, &smem);
    return {G, smem};
}

bool fed_round_small_supported(int64_t kind, int64_t din, int64_t hid, int64_t dout) {
    return fdb::fed_round_small_supported((int)kind, (int)din, (int)hid, (int)dout) != 0;
}

std::vector<Tensor> mlp_eval_matrix(Tensor theta, Tensor X, Tensor Y, Tensor nsamp, int64_t kind, int64_t din, int64_t hid, int64_t dout) {
    CHECK_CUDA_F32(theta); CHECK_CUDA_F32(X); CHECK_CUDA_I32(Y); CHECK_CUDA_I32(nsamp);
    c10::cuda::CUDAGuard guard(X.device());
    const int M = (int)theta.size(0), C = (int)X.size(0), S = (int)X.size(1);
    auto correct = torch::zeros({M, C}, theta.options());
    auto loss = torch::zeros({M, C}, theta.options());
    auto sq = torch::zeros({M, C}, theta.options());
    const int rc = fdb::mlp_eval_matrix_launch((int)kind, (int)din, (int)hid, (int)dout, theta.data_ptr<float>(), (int)theta.stride(0), M,
                                               X.data_ptr<float>(), Y.data_ptr<int>(), nsamp.data_ptr<int>(), C, S,
                                               correct.data_ptr<float>(), loss.data_ptr<float>(), sq.data_ptr<float>(), cur_stream());
    CHECK_OK(rc, "mlp_eval_matrix");
    return {correct, loss, sq};
}

// ---------------------------------------------------------------------------------- arena streaming ops
Tensor cluster_aggregate(Tensor theta, Tensor cp, Tensor n) {
    CHECK_CUDA_F32(theta); CHECK_CUDA_F32(cp); CHECK_CUDA_F32(n);
    c10::cuda::CUDAGuard guard(theta.device());
    const int C = (int)cp.size(0), M = (int)cp.size(1), P = (int)cp.size(2);
    TORCH_CHECK(theta.size(0) == M && theta.size(1) == P && theta.stride(1) == 1, "theta must be [M, P] with unit inner stride");
    auto tot = torch::zeros({M}, theta.options());
    CHECK_OK(fdb::cluster_aggregate_launch(theta.data_ptr<float>(), (int)theta.stride(0), cp.data_ptr<float>(), n.data_ptr<float>(), C, M, P,
                                           tot.data_ptr<float>(), 0, 0.f, 0.f, 0.9f, 0.999f, 1e-8f, 1, nullptr, nullptr, cur_stream()),
             "cluster_aggregate");
    return tot;
}

Tensor cluster_aggregate_opt(Tensor theta, Tensor cp, Tensor n, int64_t opt_kind, double lr, double momentum, double b1, double b2, double eps,
                             int64_t step, c10::optional<Tensor> s0, c10::optional<Tensor> s1) {
    CHECK_CUDA_F32(theta); CHECK_CUDA_F32(cp); CHECK_CUDA_F32(n);
    c10::cuda::CUDAGuard guard(theta.device());
    const int C = (int)cp.size(0), M = (int)cp.size(1), P = (int)cp.size(2);
    auto tot = torch::zeros({M}, theta.options());
    CHECK_OK(fdb::cluster_aggregate_launch(theta.data_ptr<float>(), (int)theta.stride(0), cp.data_ptr<float>(), n.data_ptr<float>(), C, M, P,
                                           tot.data_ptr<float>(), (int)opt_kind, (float)lr, (float)momentum, (float)b1, (float)b2, (float)eps,
                                           (int)step, opt_ptr<float>(s0), opt_ptr<float>(s1), cur_stream()),
             "cluster_aggregate_opt");
    return tot;
}

Tensor weighted_average(Tensor rows, Tensor w) {
    CHECK_CUDA_F32(rows); CHECK_CUDA_F32(w);
    c10::cuda::CUDAGuard guard(rows.device());
    auto out = torch::empty({rows.size(1)}, rows.options());
    CHECK_OK(fdb::weighted_average_launch(rows.data_ptr<float>(), w.data_ptr<float>(), (int)rows.size(0), rows.size(1), out.data_ptr<float>(),
                                          cur_stream()), "weighted_average");
    return out;
}

void merge_axpby(Tensor theta, int64_t base, int64_t second, double w1, double w2) {
    CHECK_CUDA_F32(theta);
    c10::cuda::CUDAGuard guard(theta.device());
    CHECK_OK(fdb::merge_axpby_launch(theta.data_ptr<float>() + base * theta.stride(0), theta.data_ptr<float>() + second * theta.stride(0),
                                     (float)w1, (float)w2, theta.size(1), cur_stream()), "merge_axpby");
}

double mean_sq_diff(Tensor a, Tensor b) {
    CHECK_CUDA_F32(a); CHECK_CUDA_F32(b);
    c10::cuda::CUDAGuard guard(a.device());
    auto out = torch::zeros({1}, a.options().dtype(torch::kFloat64));
    CHECK_OK(fdb::sq_diff_sum_launch(a.data_ptr<float>(), b.data_ptr<float>(), a.numel(), out.data_ptr<double>(), cur_stream()), "mean_sq_diff");
    return out.item<double>() / (double)a.numel();
}

Tensor gossip_mix(Tensor X, Tensor Wm) {
    CHECK_CUDA_F32(X); CHECK_CUDA_F32(Wm);
    c10::cuda::CUDAGuard guard(X.device());
    auto out = torch::empty_like(X);
    CHECK_OK(fdb::gossip_mix_launch(X.data_ptr<float>(), Wm.data_ptr<float>(), (int)X.size(0), X.size(1), out.data_ptr<float>(), cur_stream()),
             "gossip_mix");
    return out;
}

Tensor robust_clip(Tensor rows, Tensor g, double bound, c10::optional<Tensor> mask, double stddev, int64_t seed) {
    CHECK_CUDA_F32(rows); CHECK_CUDA_F32(g);
    c10::cuda::CUDAGuard guard(rows.device());
    const int R = (int)rows.size(0);
    auto scratch = torch::zeros({R}, rows.options());
    auto nrm = torch::zeros({R}, rows.options());
    CHECK_OK(fdb::robust_clip_launch(rows.data_ptr<float>(), g.data_ptr<float>(), opt_ptr<unsigned char>(mask), R, rows.size(1), (float)bound,
                                     scratch.data_ptr<float>(), nrm.data_ptr<float>(), (float)stddev, (unsigned)seed, cur_stream()), "robust_clip");
    return nrm;
}

// cp: the client arena [C_arena, M, P]; cidx: int32 [C] arena rows of this rank's clients (or None: rows 0..C-1 of cp);
// n: [C, M] weights of those clients; chunk_done: int32 [max_chunks] local counters; returns the grid size used
int64_t fedavg_reduce_apply_peer(Tensor cp, c10::optional<Tensor> cidx, Tensor n, int64_t P, int64_t theta_stride, int64_t world, int64_t rank,
                                 std::vector<int64_t> part_ptrs, std::vector<int64_t> theta_ptrs, std::vector<int64_t> tot_ptrs,
                                 std::vector<int64_t> flag_ptrs, Tensor grid_sync, Tensor chunk_done, int64_t launch_idx, int64_t epoch,
                                 int64_t grid_base, int64_t timeout_ms, Tensor error_flag, int64_t mc_part, int64_t mc_theta) {
    CHECK_CUDA_F32(cp); CHECK_CUDA_F32(n); CHECK_CUDA_I32(grid_sync); CHECK_CUDA_I32(error_flag); CHECK_CUDA_I32(chunk_done);
    c10::cuda::CUDAGuard guard(cp.device());
    const int C = (int)n.size(0), M = (int)cp.size(1);
    TORCH_CHECK(cp.dim() == 3 && cp.size(2) == P && cp.is_contiguous() && n.dim() == 2 && n.size(1) == M && n.is_contiguous(),
                "cp must be contiguous [C_arena, M, P] and n contiguous [C, M]");
    const int* ci = nullptr;
    if (cidx.has_value() && cidx->defined()) {
        CHECK_CUDA_I32(*cidx);
        TORCH_CHECK(cidx->numel() == C && cidx->is_contiguous(), "cidx must hold one arena row per local client");
        ci = cidx->data_ptr<int>();
    } else {
        TORCH_CHECK(cp.size(0) >= C, "cp has fewer rows than n");
    }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cp.device().index());
    std::vector<long long> a(part_ptrs.begin(), part_ptrs.end()), b(theta_ptrs.begin(), theta_ptrs.end()),
        c(tot_ptrs.begin(), tot_ptrs.end()), d(flag_ptrs.begin(), flag_ptrs.end());
    const int rc = fdb::fedavg_reduce_apply_peer_launch(cp.data_ptr<float>(), ci, n.data_ptr<float>(), C, M, (int)P, (int)theta_stride, (int)world,
                                                        (int)rank, a.data(), b.data(), c.data(), d.data(), (long long)mc_part, (long long)mc_theta,
                                                        reinterpret_cast<unsigned*>(grid_sync.data_ptr<int>()),
                                                        reinterpret_cast<unsigned*>(chunk_done.data_ptr<int>()), (int)chunk_done.numel(),
                                                        (unsigned)launch_idx, (unsigned)epoch, (unsigned)grid_base, sms, timeout_ms,
                                                        error_flag.data_ptr<int>(), cur_stream());
    CHECK_OK(rc, "fedavg_reduce_apply_peer");
    return sms;
}

int64_t gossip_mix_peer(std::vector<int64_t> x_ptrs, std::vector<int64_t> flag_ptrs, std::vector<double> w, int64_t P, int64_t world,
                        int64_t rank, Tensor grid_sync, int64_t grid_base, int64_t epoch, int64_t timeout_ms, Tensor error_flag) {
    CHECK_CUDA_I32(grid_sync); CHECK_CUDA_I32(error_flag);
    c10::cuda::CUDAGuard guard(grid_sync.device());
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, grid_sync.device().index());
    std::vector<long long> a(x_ptrs.begin(), x_ptrs.end()), b(flag_ptrs.begin(), flag_ptrs.end());
    std::vector<float> wf(w.begin(), w.end());
    wf.resize(8, 0.f);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(sms, (P / 4 + 511) / 512));
    const int rc = fdb::gossip_mix_peer_launch(a.data(), b.data(), wf.data(), (int)P, (int)world, (int)rank,
                                               reinterpret_cast<unsigned*>(grid_sync.data_ptr<int>()), (unsigned)grid_base, (unsigned)epoch,
                                               grid, timeout_ms, error_flag.data_ptr<int>(), cur_stream());
    CHECK_OK(rc, "gossip_mix_peer");
    return grid;
}

// ---------------------------------------------------------------------------------- evaluation reductions
void eval_logits(Tensor logits, Tensor target, Tensor acc) {
    CHECK_CUDA_F32(logits); CHECK_CUDA_I32(target); CHECK_CUDA_F32(acc);
    c10::cuda::CUDAGuard guard(logits.device());
    CHECK_OK(fdb::eval_logits_launch(logits.data_ptr<float>(), target.data_ptr<int>(), (int)logits.size(0), (int)logits.size(1),
                                     acc.data_ptr<float>(), cur_stream()), "eval_logits");
}
Tensor aue_sqerr(Tensor logits, Tensor target) {
    CHECK_CUDA_F32(logits); CHECK_CUDA_I32(target);
    c10::cuda::CUDAGuard guard(logits.device());
    auto out = torch::zeros({}, logits.options());
    CHECK_OK(fdb::aue_sqerr_launch(logits.data_ptr<float>(), target.data_ptr<int>(), (int)logits.size(0), (int)logits.size(1),
                                   out.data_ptr<float>(), cur_stream()), "aue_sqerr");
    return out;
}
Tensor ensemble_vote(Tensor preds, Tensor w, int64_t classes) {
    CHECK_CUDA_I32(preds); CHECK_CUDA_F32(w);
    c10::cuda::CUDAGuard guard(preds.device());
    auto out = torch::empty({preds.size(1)}, preds.options());
    CHECK_OK(fdb::ensemble_vote_launch(preds.data_ptr<int>(), w.data_ptr<float>(), (int)preds.size(0), (int)preds.size(1), (int)classes,
                                       out.data_ptr<int>(), cur_stream()), "ensemble_vote");
    return out.to(torch::kInt64);
}
Tensor confusion_matrix(Tensor pred, Tensor target, int64_t classes) {
    CHECK_CUDA_I32(pred); CHECK_CUDA_I32(target);
    c10::cuda::CUDAGuard guard(pred.device());
    auto out = torch::zeros({classes, classes}, pred.options());
    CHECK_OK(fdb::confusion_matrix_launch(pred.data_ptr<int>(), target.data_ptr<int>(), (int)pred.numel(), (int)classes, out.data_ptr<int>(),
                                          cur_stream()), "confusion_matrix");
    return out;
}

// ---------------------------------------------------------------------------------- optimizers
void adam_amsgrad_rows(Tensor p, Tensor g, Tensor m, Tensor v, Tensor vmax, Tensor steps, double lr, double wd, double b1, double b2, double eps,
                       c10::optional<Tensor> row_mask) {
    CHECK_CUDA_F32(p); CHECK_CUDA_F32(g); CHECK_CUDA_F32(m); CHECK_CUDA_F32(v); CHECK_CUDA_F32(vmax); CHECK_CUDA_I32(steps);
    c10::cuda::CUDAGuard guard(p.device());
    TORCH_CHECK(p.is_contiguous() && m.is_contiguous() && v.is_contiguous() && vmax.is_contiguous(), "arena rows must be contiguous");
    const int R = (int)steps.numel();
    const long long P = p.numel() / R;
    CHECK_OK(fdb::adam_amsgrad_rows_launch(p.data_ptr<float>(), g.data_ptr<float>(), m.data_ptr<float>(), v.data_ptr<float>(),
                                           vmax.data_ptr<float>(), steps.data_ptr<int>(), opt_ptr<unsigned char>(row_mask), R, P, (float)lr,
                                           (float)wd, (float)b1, (float)b2, (float)eps, cur_stream()), "adam_amsgrad_rows");
}
void sgd_rows(Tensor p, Tensor g, double lr, double wd) {
    CHECK_CUDA_F32(p); CHECK_CUDA_F32(g);
    c10::cuda::CUDAGuard guard(p.device());
    CHECK_OK(fdb::sgd_rows_launch(p.data_ptr<float>(), g.data_ptr<float>(), p.numel(), (float)lr, (float)wd, cur_stream()), "sgd_rows");
}

// ---------------------------------------------------------------------------------- clustering geometry / MPC / misc
std::vector<Tensor> gram_cosine(Tensor U, double eps) {
    CHECK_CUDA_F32(U);
    c10::cuda::CUDAGuard guard(U.device());
    const int n = (int)U.size(0);
    auto S = torch::empty({n, n}, U.options().dtype(torch::kFloat64));
    auto nrm = torch::empty({n}, U.options().dtype(torch::kFloat64));
    auto part = torch::empty({fdb::gram_workspace_doubles()}, S.options());   // caching allocator: no driver call on the hot path
    const int rc = fdb::gram_launch(U.data_ptr<float>(), n, U.size(1), eps, S.data_ptr<double>(), nrm.data_ptr<double>(),
                                    part.data_ptr<double>(), cur_stream());
    if (rc == -5) {  // > 32 rows: library GEMM (cold path)
        auto G = torch::matmul(U.to(torch::kFloat64), U.to(torch::kFloat64).t());
        nrm = torch::sqrt(torch::diagonal(G));
        S = G / (nrm.unsqueeze(1) * nrm.unsqueeze(0) + eps);
    } else {
        CHECK_OK(rc, "gram");
    }
    return {S, nrm};
}

Tensor modp_matmul(Tensor A, Tensor B, int64_t p) {
    TORCH_CHECK(A.is_cuda() && A.scalar_type() == torch::kInt64 && B.scalar_type() == torch::kInt64, "modp_matmul needs CUDA int64");
    c10::cuda::CUDAGuard guard(A.device());
    auto C = torch::empty({A.size(0), B.size(1)}, A.options());
    CHECK_OK(fdb::modp_matmul_launch(reinterpret_cast<const long long*>(A.data_ptr<int64_t>()), reinterpret_cast<const long long*>(B.data_ptr<int64_t>()),
                                     reinterpret_cast<long long*>(C.data_ptr<int64_t>()), (int)A.size(0), (int)A.size(1), (int)B.size(1), p,
                                     cur_stream()), "modp_matmul");
    return C;
}

std::vector<Tensor> kd_kl_fwd_bwd(Tensor s, Tensor t, double T) {
    CHECK_CUDA_F32(s); CHECK_CUDA_F32(t);
    c10::cuda::CUDAGuard guard(s.device());
    auto loss = torch::zeros({}, s.options());
    auto grad = torch::empty_like(s);
    CHECK_OK(fdb::kd_kl_launch(s.data_ptr<float>(), t.data_ptr<float>(), (int)s.size(0), (int)s.size(1), (float)T, loss.data_ptr<float>(),
                               grad.data_ptr<float>(), cur_stream()), "kd_kl");
    return {loss, grad};
}

std::vector<Tensor> vfl_bce_grad(Tensor parts, Tensor y) {
    CHECK_CUDA_F32(parts); CHECK_CUDA_F32(y);
    c10::cuda::CUDAGuard guard(parts.device());
    const int K = (int)parts.size(0), B = (int)parts.size(1);
    auto loss = torch::zeros({}, parts.options());
    auto grad = torch::empty({B, 1}, parts.options());
    CHECK_OK(fdb::vfl_bce_launch(parts.data_ptr<float>(), y.data_ptr<float>(), K, B, loss.data_ptr<float>(), grad.data_ptr<float>(), cur_stream()),
             "vfl_bce");
    return {loss, grad};
}

Tensor group_norm_fwd(Tensor x, int64_t groups, c10::optional<Tensor> w, c10::optional<Tensor> b, double eps) {
    CHECK_CUDA_F32(x);
    c10::cuda::CUDAGuard guard(x.device());
    auto y = torch::empty_like(x);
    const int N = (int)x.size(0), C = (int)x.size(1);
    const int HW = (int)(x.numel() / ((int64_t)N * C));
    CHECK_OK(fdb::group_norm_fwd_launch(x.data_ptr<float>(), y.data_ptr<float>(), opt_ptr<float>(w), opt_ptr<float>(b), N, C, HW, (int)groups,
                                        (float)eps, cur_stream()), "group_norm_fwd");
    return y;
}

// training forward: also returns the per-(sample, group) mean / rstd the backward kernel needs
std::vector<Tensor> group_norm_fwd_train(Tensor x, int64_t groups, c10::optional<Tensor> w, c10::optional<Tensor> b, double eps) {
    CHECK_CUDA_F32(x);
    TORCH_CHECK(x.is_contiguous(), "group_norm: x must be contiguous NCHW");
    c10::cuda::CUDAGuard guard(x.device());
    auto y = torch::empty_like(x);
    const int N = (int)x.size(0), C = (int)x.size(1);
    const int HW = (int)(x.numel() / ((int64_t)N * C));
    auto mean = torch::empty({N * groups}, x.options());
    auto rstd = torch::empty({N * groups}, x.options());
    CHECK_OK(fdb::group_norm_fwd_launch(x.data_ptr<float>(), y.data_ptr<float>(), opt_ptr<float>(w), opt_ptr<float>(b), N, C, HW, (int)groups,
                                        (float)eps, cur_stream(), mean.data_ptr<float>(), rstd.data_ptr<float>()), "group_norm_fwd");
    return {y, mean, rstd};
}
// -> (dx, dgamma [C], dbeta [C])
// Training-mode BatchNorm over a channels_last activation given as its NHWC view x [..., C] (misc.cu::bn_nhwc_*): the running
// statistics are updated in place; -> (y, mean, rstd)
std::vector<Tensor> bn_nhwc_fwd(Tensor x, Tensor y, c10::optional<Tensor> w, c10::optional<Tensor> b, c10::optional<Tensor> run_mean,
                                c10::optional<Tensor> run_var, double eps, double momentum) {
    CHECK_CUDA_F32(x); CHECK_CUDA_F32(y);
    TORCH_CHECK(x.is_contiguous() && x.dim() >= 2 && y.is_contiguous() && y.sizes() == x.sizes(), "bn_nhwc_fwd: contiguous [..., C] input / output");
    c10::cuda::CUDAGuard guard(x.device());
    const int C = (int)x.size(-1);
    const long long rows = x.numel() / C;
    auto mean = torch::empty({C}, x.options()), rstd = torch::empty({C}, x.options()), sums = torch::empty({2, C}, x.options());
    Tensor wc, bc;
    if (w.has_value() && w->defined()) { wc = w->contiguous(); TORCH_CHECK(wc.numel() == C && wc.scalar_type() == torch::kFloat32, "bn weight"); }
    if (b.has_value() && b->defined()) { bc = b->contiguous(); TORCH_CHECK(bc.numel() == C && bc.scalar_type() == torch::kFloat32, "bn bias"); }
    float *rm = nullptr, *rv = nullptr;
    if (run_mean.has_value() && run_mean->defined()) {
        TORCH_CHECK(run_var.has_value() && run_mean->is_contiguous() && run_var->is_contiguous() && run_mean->numel() == C && run_var->numel() == C, "bn running stats");
        rm = run_mean->data_ptr<float>(); rv = run_var->data_ptr<float>();
    }
    CHECK_OK(fdb::bn_nhwc_fwd_launch(x.data_ptr<float>(), wc.defined() ? wc.data_ptr<float>() : nullptr, bc.defined() ? bc.data_ptr<float>() : nullptr,
                                     y.data_ptr<float>(), mean.data_ptr<float>(), rstd.data_ptr<float>(), rm, rv, sums.data_ptr<float>(), rows, C,
                                     (float)eps, (float)momentum, cur_stream()), "bn_nhwc_fwd");
    return {mean, rstd};
}
// -> (dx, dweight, dbias)
std::vector<Tensor> bn_nhwc_bwd(Tensor x, Tensor dy, c10::optional<Tensor> w, Tensor mean, Tensor rstd) {
    CHECK_CUDA_F32(x); CHECK_CUDA_F32(dy);
    TORCH_CHECK(x.is_contiguous() && dy.is_contiguous() && x.sizes() == dy.sizes(), "bn_nhwc_bwd: contiguous x / dy of equal shape");
    c10::cuda::CUDAGuard guard(x.device());
    const int C = (int)x.size(-1);
    const long long rows = x.numel() / C;
    auto dx = torch::empty_like(x);
    auto dw = torch::empty({C}, x.options()), db = torch::empty({C}, x.options()), sums = torch::empty({2, C}, x.options());
    Tensor wc;
    if (w.has_value() && w->defined()) wc = w->contiguous();
    CHECK_OK(fdb::bn_nhwc_bwd_launch(x.data_ptr<float>(), dy.data_ptr<float>(), wc.defined() ? wc.data_ptr<float>() : nullptr, mean.data_ptr<float>(),
                                     rstd.data_ptr<float>(), dx.data_ptr<float>(), dw.data_ptr<float>(), db.data_ptr<float>(), sums.data_ptr<float>(),
                                     rows, C, cur_stream()), "bn_nhwc_bwd");
    return {dx, dw, db};
}
std::vector<Tensor> group_norm_bwd(Tensor x, Tensor dy, c10::optional<Tensor> w, Tensor mean, Tensor rstd, int64_t groups) {
    CHECK_CUDA_F32(x); CHECK_CUDA_F32(dy); CHECK_CUDA_F32(mean); CHECK_CUDA_F32(rstd);
    TORCH_CHECK(x.is_contiguous() && dy.is_contiguous() && x.sizes() == dy.sizes(), "group_norm_bwd: contiguous x / dy of equal shape");
    c10::cuda::CUDAGuard guard(x.device());
    const int N = (int)x.size(0), C = (int)x.size(1);
    const int HW = (int)(x.numel() / ((int64_t)N * C));
    auto dx = torch::empty_like(x);
    auto dg = torch::empty({N, C}, x.options());
    auto db = torch::empty({N, C}, x.options());
    CHECK_OK(fdb::group_norm_bwd_launch(x.data_ptr<float>(), dy.data_ptr<float>(), opt_ptr<float>(w), mean.data_ptr<float>(), rstd.data_ptr<float>(),
                                        dx.data_ptr<float>(), dg.data_ptr<float>(), db.data_ptr<float>(), N, C, HW, (int)groups, cur_stream()),
             "group_norm_bwd");
    return {dx, dg.sum(0), db.sum(0)};
}

Tensor gemm_tn_bias_act(Tensor A, Tensor B, c10::optional<Tensor> bias, bool relu, bool out_fp32) {
    TORCH_CHECK(A.is_cuda() && A.scalar_type() == torch::kBFloat16 && B.scalar_type() == torch::kBFloat16, "gemm_tn needs CUDA bf16 operands");
    TORCH_CHECK(A.is_contiguous() && B.is_contiguous() && A.size(1) == B.size(1), "gemm_tn: A [M,K], B [N,K] contiguous");
    c10::cuda::CUDAGuard guard(A.device());
    const int M = (int)A.size(0), K = (int)A.size(1), N = (int)B.size(0);
    auto D = torch::empty({M, N}, A.options().dtype(out_fp32 ? torch::kFloat32 : torch::kBFloat16));
    const float* bp = nullptr;
    Tensor bias_f;
    if (bias.has_value() && bias->defined()) { bias_f = bias->to(torch::kFloat32).contiguous(); bp = bias_f.data_ptr<float>(); }
    Tensor ws;   // fp32 split-K accumulator for bf16 outputs, from the caching allocator
    if (!out_fp32 && fdb::gemm_split_count(M, N, K) > 1) ws = torch::empty({M, N}, A.options().dtype(torch::kFloat32));
    const int rc = fdb::gemm_launch(A.data_ptr(), B.data_ptr(), D.data_ptr(), bp, M, N, K, 0, 0, relu ? 1 : 0, out_fp32 ? 1 : 0, cur_stream(),
                                    ws.defined() ? ws.data_ptr<float>() : nullptr);
    CHECK_OK(rc, "gemm_tn (tcgen05)");
    return D;
}

// General operand layouts: A is [M,K] (a_mn = false) or [K,M] (a_mn = true); B is [N,K] (b_mn = false) or [K,N] (b_mn = true);
// D[M,N] = act(A·B + bias) with the reduction over K.  Lets the backward GEMMs consume row-major tensors without transposes.
Tensor gemm_bias_act(Tensor A, Tensor B, bool a_mn, bool b_mn, c10::optional<Tensor> bias, bool relu, bool out_fp32) {
    TORCH_CHECK(A.is_cuda() && A.scalar_type() == torch::kBFloat16 && B.scalar_type() == torch::kBFloat16, "gemm needs CUDA bf16 operands");
    TORCH_CHECK(A.is_contiguous() && B.is_contiguous() && A.dim() == 2 && B.dim() == 2, "gemm: contiguous 2-D operands");
    c10::cuda::CUDAGuard guard(A.device());
    const int M = (int)A.size(a_mn ? 1 : 0), K = (int)A.size(a_mn ? 0 : 1), N = (int)B.size(b_mn ? 1 : 0);
    TORCH_CHECK(B.size(b_mn ? 0 : 1) == K, "gemm: reduction lengths differ");
    auto D = torch::empty({M, N}, A.options().dtype(out_fp32 ? torch::kFloat32 : torch::kBFloat16));
    const float* bp = nullptr;
    Tensor bias_f;
    if (bias.has_value() && bias->defined()) { bias_f = bias->to(torch::kFloat32).contiguous(); bp = bias_f.data_ptr<float>(); }
    Tensor ws;
    if (!out_fp32 && fdb::gemm_split_count(M, N, K) > 1) ws = torch::empty({M, N}, A.options().dtype(torch::kFloat32));
    const int rc = fdb::gemm_launch(A.data_ptr(), B.data_ptr(), D.data_ptr(), bp, M, N, K, a_mn ? 1 : 0, b_mn ? 1 : 0, relu ? 1 : 0,
                                    out_fp32 ? 1 : 0, cur_stream(), ws.defined() ? ws.data_ptr<float>() : nullptr);
    CHECK_OK(rc, "gemm (tcgen05)");
    return D;
}

// Batched weight-gradient GEMM (one launch for every pair): D[bt] [M, N] fp32 = A'[rows a_k0 + bt·a_kstride …+K, M]ᵀ · B'[rows b_k0 + bt·b_kstride …+K, N]
Tensor gemm_batched_mn(Tensor A, Tensor B, int64_t K, int64_t batch, int64_t a_k0, int64_t a_kstride, int64_t b_k0, int64_t b_kstride) {
    TORCH_CHECK(A.is_cuda() && A.scalar_type() == torch::kBFloat16 && B.scalar_type() == torch::kBFloat16, "gemm_batched_mn needs CUDA bf16 operands");
    TORCH_CHECK(A.is_contiguous() && B.is_contiguous() && A.dim() == 2 && B.dim() == 2, "gemm_batched_mn: contiguous 2-D operands");
    TORCH_CHECK(a_k0 + (batch - 1) * a_kstride + K <= A.size(0) && b_k0 + (batch - 1) * b_kstride + K <= B.size(0), "gemm_batched_mn: K range");
    c10::cuda::CUDAGuard guard(A.device());
    const int M = (int)A.size(1), N = (int)B.size(1);
    auto D = torch::empty({batch, M, N}, A.options().dtype(torch::kFloat32));
    const int rc = fdb::gemm_batched_mn_launch(A.data_ptr(), B.data_ptr(), D.data_ptr<float>(), M, N, (int)K, (int)batch, (int)A.size(0),
                                               (int)B.size(0), (int)a_k0, (int)a_kstride, (int)b_k0, (int)b_kstride, cur_stream());
    CHECK_OK(rc, "gemm_batched_mn (tcgen05)");
    return D;
}

// K2 (consumer-pull broadcast): the weight matrix B[N,K] stays in the OWNER GPU's symmetric-memory arena; `b_ptr` is
// the peer-mapped device pointer.  The TMA producer of the GEMM pulls B tiles straight over NVLink inside the tile loop,
// so "broadcast the model, then run the first layer" is one kernel and no local copy of the weights ever exists.
Tensor gemm_tn_bias_act_peer(Tensor A, int64_t b_ptr, int64_t N, c10::optional<Tensor> bias, bool relu, bool out_fp32) {
    TORCH_CHECK(A.is_cuda() && A.scalar_type() == torch::kBFloat16 && A.is_contiguous(), "gemm_tn_peer: A must be CUDA bf16 [M,K]");
    TORCH_CHECK(b_ptr != 0 && N > 0, "gemm_tn_peer: null weight pointer");
    c10::cuda::CUDAGuard guard(A.device());
    const int M = (int)A.size(0), K = (int)A.size(1);
    auto D = torch::empty({M, N}, A.options().dtype(out_fp32 ? torch::kFloat32 : torch::kBFloat16));
    const float* bp = nullptr;
    Tensor bias_f;
    if (bias.has_value() && bias->defined()) { bias_f = bias->to(torch::kFloat32).contiguous(); bp = bias_f.data_ptr<float>(); }
    Tensor ws;
    if (!out_fp32 && fdb::gemm_split_count(M, (int)N, K) > 1) ws = torch::empty({M, N}, A.options().dtype(torch::kFloat32));
    const int rc = fdb::gemm_launch(A.data_ptr(), reinterpret_cast<const void*>(b_ptr), D.data_ptr(), bp, M, (int)N, K, 0, 0, relu ? 1 : 0,
                                    out_fp32 ? 1 : 0, cur_stream(), ws.defined() ? ws.data_ptr<float>() : nullptr);
    CHECK_OK(rc, "gemm_tn_peer (tcgen05)");
    return D;
}

// conv-as-GEMM helpers (csrc/conv_im2col.cu): x may be NCHW or channels_last — strides are passed through
Tensor im2col_bf16(Tensor x, int64_t kh, int64_t kw, int64_t sh, int64_t sw, int64_t ph, int64_t pw) {
    CHECK_CUDA_F32(x);
    TORCH_CHECK(x.dim() == 4, "im2col: x must be [B, C, H, W]");
    c10::cuda::CUDAGuard guard(x.device());
    const int B = (int)x.size(0), C = (int)x.size(1), H = (int)x.size(2), W = (int)x.size(3);
    const int Ho = (int)((H + 2 * ph - kh) / sh + 1), Wo = (int)((W + 2 * pw - kw) / sw + 1);
    auto cols = torch::empty({(int64_t)B * Ho * Wo, (int64_t)C * kh * kw}, x.options().dtype(torch::kBFloat16));
    CHECK_OK(fdb::im2col_bf16_launch(x.data_ptr<float>(), cols.data_ptr(), B, C, H, W, (int)kh, (int)kw, (int)sh, (int)sw, (int)ph, (int)pw,
                                     Ho, Wo, x.stride(0), x.stride(1), x.stride(2), x.stride(3), cur_stream()), "im2col");
    return cols;
}
Tensor col2im(Tensor dcols, int64_t B, int64_t C, int64_t H, int64_t W, int64_t kh, int64_t kw, int64_t sh, int64_t sw, int64_t ph,
              int64_t pw) {
    CHECK_CUDA_F32(dcols);
    c10::cuda::CUDAGuard guard(dcols.device());
    const int Ho = (int)((H + 2 * ph - kh) / sh + 1), Wo = (int)((W + 2 * pw - kw) / sw + 1);
    TORCH_CHECK(dcols.is_contiguous() && dcols.size(0) == B * Ho * Wo && dcols.size(1) == C * kh * kw, "col2im: bad dcols shape");
    auto dx = torch::empty({B, C, H, W}, dcols.options());
    CHECK_OK(fdb::col2im_launch(dcols.data_ptr<float>(), dx.data_ptr<float>(), (int)B, (int)C, (int)H, (int)W, (int)kh, (int)kw, (int)sh,
                                (int)sw, (int)ph, (int)pw, Ho, Wo, cur_stream()), "col2im");
    return dx;
}

// Launch an instantiated CUDA graph on the current stream and (optionally) wait for it, with the GIL released: the
// end-to-end round path calls this once per round instead of CUDAGraph.replay() + Stream.synchronize() (two Python →
// C++ round trips).  `exec` is `torch.cuda.CUDAGraph.raw_cuda_graph_exec()`.
void graph_launch_sync(int64_t exec, bool sync) {
    cudaStream_t stream = cur_stream();
    pybind11::gil_scoped_release nogil;
    cudaError_t e = cudaGraphLaunch(reinterpret_cast<cudaGraphExec_t>(exec), stream);
    if (e == cudaSuccess && sync) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {
        pybind11::gil_scoped_acquire gil;
        TORCH_CHECK(false, "graph_launch_sync: ", cudaGetErrorString(e));
    }
}

// ---------------------------------------------------------------------------------- persistent LSTM (lstm_tc.cu)
// offs = {emb, w_ih1, w_hh1, b_ih1, b_hh1, w_ih2, w_hh2, b_ih2, b_hh2} element offsets inside a parameter row.
static fdb::LstmArgs lstm_args(const Tensor& params, const Tensor& row_off, const std::vector<int64_t>& offs, const Tensor& tokens,
                               const c10::optional<Tensor>& gates, const c10::optional<Tensor>& cst, const c10::optional<Tensor>& hhist,
                               const Tensor& hlast, int64_t E) {
    CHECK_CUDA_F32(params); CHECK_CUDA_I32(tokens); CHECK_CUDA_F32(hlast);
    TORCH_CHECK(row_off.is_cuda() && row_off.scalar_type() == torch::kInt64, "row_off must be a CUDA int64 tensor");
    TORCH_CHECK(offs.size() == 9, "need 9 parameter offsets");
    TORCH_CHECK(tokens.dim() == 3 && tokens.size(1) == 16 && tokens.is_contiguous(), "tokens must be [npairs, 16, T] contiguous");
    const int64_t np = tokens.size(0), T = tokens.size(2);
    TORCH_CHECK(row_off.numel() == np && E >= 1 && E <= 16 && T >= 1, "lstm2: bad sizes");
    TORCH_CHECK(hlast.numel() == np * 16 * 256, "lstm2: hlast size");
    fdb::LstmArgs a{};
    a.params = params.data_ptr<float>();
    a.row_off = reinterpret_cast<const long long*>(row_off.data_ptr<int64_t>());
    a.off_emb = offs[0]; a.off_wih1 = offs[1]; a.off_whh1 = offs[2]; a.off_bih1 = offs[3]; a.off_bhh1 = offs[4];
    a.off_wih2 = offs[5]; a.off_whh2 = offs[6]; a.off_bih2 = offs[7]; a.off_bhh2 = offs[8];
    a.tokens = tokens.data_ptr<int>();
    if (gates.has_value() && gates->defined()) {
        TORCH_CHECK(cst.has_value() && cst->defined(), "lstm2: gates and cst come together");
        CHECK_CUDA_F32(*gates); CHECK_CUDA_F32(*cst);
        TORCH_CHECK(gates->numel() == np * 2 * T * 16 * 1024 && cst->numel() == np * 2 * T * 16 * 256, "lstm2: workspace sizes");
        a.gates = gates->data_ptr<float>(); a.cst = cst->data_ptr<float>();
    }
    if (hhist.has_value() && hhist->defined()) {
        TORCH_CHECK(hhist->is_cuda() && hhist->scalar_type() == torch::kBFloat16 && hhist->numel() == np * 2 * (T + 1) * 16 * 256,
                    "hhist must be CUDA bf16 [2, npairs, T+1, 16, 256]");
        a.hhist = hhist->data_ptr();
    }
    a.hlast = hlast.data_ptr<float>();
    a.T = (int)T; a.E = (int)E;
    return a;
}

void lstm2_forward(Tensor params, Tensor row_off, std::vector<int64_t> offs, Tensor tokens, c10::optional<Tensor> gates,
                   c10::optional<Tensor> cst, c10::optional<Tensor> hhist, Tensor hlast, int64_t E, c10::optional<Tensor> dbg) {
    c10::cuda::CUDAGuard guard(params.device());
    fdb::LstmArgs a = lstm_args(params, row_off, offs, tokens, gates, cst, hhist, hlast, E);
    if (dbg.has_value() && dbg->defined()) {
        TORCH_CHECK(dbg->is_cuda() && dbg->scalar_type() == torch::kInt64 && dbg->numel() >= 8, "dbg must be a CUDA int64[8] tensor");
        a.dbg = reinterpret_cast<long long*>(dbg->data_ptr<int64_t>());
    }
    CHECK_OK(fdb::lstm2_fwd_launch(a, (int)tokens.size(0), cur_stream()), "lstm2_fwd (tcgen05 cluster kernel)");
}

void lstm2_backward(Tensor params, Tensor row_off, std::vector<int64_t> offs, Tensor tokens, Tensor gates, Tensor cst, Tensor hhist,
                    Tensor hlast, int64_t E, c10::optional<Tensor> dh2_last, c10::optional<Tensor> dh2_all, Tensor dgates) {
    c10::cuda::CUDAGuard guard(params.device());
    fdb::LstmArgs a = lstm_args(params, row_off, offs, tokens, gates, cst, hhist, hlast, E);
    TORCH_CHECK(a.gates != nullptr, "lstm2_backward needs the forward history");
    const int64_t np = tokens.size(0), T = tokens.size(2);
    TORCH_CHECK(dgates.is_cuda() && dgates.scalar_type() == torch::kBFloat16 && dgates.numel() == np * 2 * T * 16 * 1024, "dgates workspace");
    if (dh2_all.has_value() && dh2_all->defined()) {
        CHECK_CUDA_F32(*dh2_all);
        TORCH_CHECK(dh2_all->numel() == np * T * 16 * 256 && dh2_all->is_contiguous(), "dh2_all must be [npairs, T, 16, 256]");
        a.dh2_all = dh2_all->data_ptr<float>();
    } else {
        TORCH_CHECK(dh2_last.has_value() && dh2_last->defined(), "lstm2_backward needs dh2_last or dh2_all");
        CHECK_CUDA_F32(*dh2_last);
        TORCH_CHECK(dh2_last->numel() == np * 16 * 256 && dh2_last->is_contiguous(), "dh2_last must be [npairs, 16, 256]");
        a.dh2_last = dh2_last->data_ptr<float>();
    }
    a.dgates = dgates.data_ptr();
    CHECK_OK(fdb::lstm2_bwd_launch(a, (int)np, cur_stream()), "lstm2_bwd (tcgen05 cluster kernel)");
}

// fc + softmax-CE + all head gradients for `nchunks` 16-row chunks (lstm_tc.cu::lstm_head_kernel)
void lstm_head(Tensor params, Tensor row_off, int64_t off_fcw, int64_t off_fcb, Tensor hlast, Tensor labels, Tensor scale, Tensor dh,
               Tensor dW, Tensor db, c10::optional<Tensor> loss, int64_t V) {
    CHECK_CUDA_F32(params); CHECK_CUDA_F32(hlast); CHECK_CUDA_I32(labels); CHECK_CUDA_F32(scale); CHECK_CUDA_F32(dh); CHECK_CUDA_F32(dW);
    CHECK_CUDA_F32(db);
    TORCH_CHECK(row_off.is_cuda() && row_off.scalar_type() == torch::kInt64, "row_off must be a CUDA int64 tensor");
    c10::cuda::CUDAGuard guard(params.device());
    const int64_t n = row_off.numel();
    TORCH_CHECK(hlast.numel() == n * 16 * 256 && labels.numel() == n * 16 && scale.numel() == n && dh.numel() == n * 16 * 256 &&
                dW.numel() == n * V * 256 && db.numel() == n * V, "lstm_head: tensor sizes");
    fdb::LstmHeadArgs a{};
    a.params = params.data_ptr<float>();
    a.row_off = reinterpret_cast<const long long*>(row_off.data_ptr<int64_t>());
    a.off_fcw = off_fcw; a.off_fcb = off_fcb;
    a.hlast = hlast.data_ptr<float>(); a.labels = labels.data_ptr<int>(); a.scale = scale.data_ptr<float>();
    a.dh = dh.data_ptr<float>(); a.dW = dW.data_ptr<float>(); a.db = db.data_ptr<float>();
    a.loss = opt_ptr<float>(loss);
    a.V = (int)V;
    CHECK_OK(fdb::lstm_head_launch(a, (int)n, cur_stream()), "lstm_head");
}

// ---------------------------------------------------------------------------------- implicit-GEMM convolution (conv_igemm.cu)
// x: NHWC fp32 [N, H, W, C]; wq: packed bf16 [K][R][S][C]; -> y NHWC fp32 [N, P, Q, K] = act(conv(x, w) + bias)
Tensor conv_igemm_fwd(Tensor x, Tensor wq, c10::optional<Tensor> bias, int64_t stride, int64_t pad_h, int64_t pad_w, bool relu) {
    CHECK_CUDA_F32(x);
    TORCH_CHECK(x.dim() == 4 && x.is_contiguous(), "conv_igemm: x must be contiguous NHWC");
    TORCH_CHECK(wq.is_cuda() && wq.scalar_type() == torch::kBFloat16 && wq.dim() == 4 && wq.is_contiguous(), "conv_igemm: wq must be packed bf16 [K,R,S,C]");
    const int N = (int)x.size(0), H = (int)x.size(1), W = (int)x.size(2), C = (int)x.size(3);
    const int K = (int)wq.size(0), R = (int)wq.size(1), S = (int)wq.size(2);
    TORCH_CHECK(wq.size(3) == C, "conv_igemm: channel mismatch");
    TORCH_CHECK(C % 16 == 0 && K % 32 == 0, "conv_igemm forward needs Cin % 16 == 0 and Cout % 32 == 0 (got ", C, ", ", K, ")");
    const int P = (H + 2 * (int)pad_h - R) / (int)stride + 1, Q = (W + 2 * (int)pad_w - S) / (int)stride + 1;
    c10::cuda::CUDAGuard guard(x.device());
    auto y = torch::empty({N, P, Q, K}, x.options());
    Tensor bias_f;
    fdb::ConvArgs a{};
    a.x = x.data_ptr<float>(); a.wq = reinterpret_cast<const __nv_bfloat16*>(wq.data_ptr()); a.y = y.data_ptr<float>();
    if (bias.has_value() && bias->defined()) { bias_f = bias->to(torch::kFloat32).contiguous(); a.bias = bias_f.data_ptr<float>(); }
    a.N = N; a.H = H; a.W = W; a.C = C; a.Kout = K; a.R = R; a.S = S; a.P = P; a.Q = Q;
    a.pad_h = (int)pad_h; a.pad_w = (int)pad_w; a.stride = (int)stride; a.mode = 0; a.relu = relu ? 1 : 0;
    CHECK_OK(fdb::conv_igemm_launch(a, cur_stream()), "conv_igemm forward (tcgen05)");
    return y;
}
// dy: NHWC fp32 [N, P, Q, K]; wq_t: packed bf16 [C][R][S][K]; -> dx NHWC fp32 [N, H, W, C]
Tensor conv_igemm_dgrad(Tensor dy, Tensor wq_t, int64_t H, int64_t W, int64_t stride, int64_t pad_h, int64_t pad_w) {
    CHECK_CUDA_F32(dy);
    TORCH_CHECK(dy.dim() == 4 && dy.is_contiguous(), "conv_igemm_dgrad: dy must be contiguous NHWC");
    TORCH_CHECK(wq_t.is_cuda() && wq_t.scalar_type() == torch::kBFloat16 && wq_t.dim() == 4 && wq_t.is_contiguous(), "conv_igemm_dgrad: wq_t must be packed bf16 [C,R,S,K]");
    const int N = (int)dy.size(0), P = (int)dy.size(1), Q = (int)dy.size(2), K = (int)dy.size(3);
    const int C = (int)wq_t.size(0), R = (int)wq_t.size(1), S = (int)wq_t.size(2);
    TORCH_CHECK(wq_t.size(3) == K, "conv_igemm_dgrad: channel mismatch");
    TORCH_CHECK(K % 16 == 0 && C % 32 == 0, "conv_igemm dgrad needs Cout % 16 == 0 and Cin % 32 == 0 (got ", K, ", ", C, ")");
    c10::cuda::CUDAGuard guard(dy.device());
    auto dx = torch::empty({N, H, W, C}, dy.options());
    fdb::ConvArgs a{};
    a.x = dy.data_ptr<float>(); a.wq = reinterpret_cast<const __nv_bfloat16*>(wq_t.data_ptr()); a.y = dx.data_ptr<float>();
    a.N = N; a.H = P; a.W = Q; a.C = K; a.Kout = C; a.R = R; a.S = S; a.P = (int)H; a.Q = (int)W;
    a.pad_h = (int)pad_h; a.pad_w = (int)pad_w; a.stride = (int)stride; a.mode = 1; a.relu = 0;
    CHECK_OK(fdb::conv_igemm_launch(a, cur_stream()), "conv_igemm dgrad (tcgen05)");
    return dx;
}
// x: NHWC fp32 [N, H, W, C]; dy: NHWC fp32 [N, P, Q, K]; -> dW fp32 OIHW [K, C, R, S]
// `accum_into`: an existing fp32 OIHW gradient buffer to ADD into (no zero-fill, no extra accumulate kernel) — the federated
// executor's parameters already own a zeroed `.grad` view of the flat gradient row
Tensor conv_igemm_wgrad(Tensor x, Tensor dy, int64_t R, int64_t S, int64_t stride, int64_t pad_h, int64_t pad_w, c10::optional<Tensor> accum_into,
                        bool ohwi) {
    CHECK_CUDA_F32(x); CHECK_CUDA_F32(dy);
    TORCH_CHECK(x.is_contiguous() && dy.is_contiguous() && x.dim() == 4 && dy.dim() == 4, "conv_igemm_wgrad: contiguous NHWC tensors");
    TORCH_CHECK(x.size(3) % 8 == 0 && dy.size(3) % 32 == 0, "conv_igemm wgrad needs Cin % 8 == 0 and Cout % 32 == 0");
    c10::cuda::CUDAGuard guard(x.device());
    const int N = (int)x.size(0), H = (int)x.size(1), W = (int)x.size(2), C = (int)x.size(3);
    const int P = (int)dy.size(1), Q = (int)dy.size(2), K = (int)dy.size(3);
    Tensor dw;
    if (accum_into.has_value() && accum_into->defined()) {
        dw = *accum_into;
        CHECK_CUDA_F32(dw);
        TORCH_CHECK(dw.is_contiguous() && dw.numel() == (int64_t)K * C * R * S, "conv_igemm_wgrad: accum_into must be a contiguous OIHW buffer");
    } else {
        dw = ohwi ? torch::empty({K, R, S, C}, x.options()) : torch::empty({K, C, R, S}, x.options());
        cudaMemsetAsync(dw.data_ptr<float>(), 0, (size_t)dw.numel() * sizeof(float), cur_stream());
    }
    fdb::ConvArgs a{};
    a.mode = ohwi ? 1 : 0;       // layout of dw: [K][R][S][C] (channels_last storage of the parameter) or OIHW
    a.x = x.data_ptr<float>(); a.dy = dy.data_ptr<float>(); a.dw = dw.data_ptr<float>();
    a.N = N; a.H = H; a.W = W; a.C = C; a.Kout = K; a.R = (int)R; a.S = (int)S; a.P = P; a.Q = Q;
    a.pad_h = (int)pad_h; a.pad_w = (int)pad_w; a.stride = (int)stride;
    CHECK_OK(fdb::conv_wgrad_launch(a, cur_stream()), "conv_igemm wgrad (tcgen05)");
    return dw;
}

// ---- TMA-im2col path (gemm_tc.cu): bf16 NHWC operands, the GEMM mainloop's producer fetches im2col boxes with the TMA unit
Tensor conv_cast_bf16(Tensor x, c10::optional<Tensor> gate) {
    CHECK_CUDA_F32(x);
    TORCH_CHECK(x.is_contiguous(), "conv_cast_bf16: contiguous input");
    c10::cuda::CUDAGuard guard(x.device());
    const float* g = nullptr;
    if (gate.has_value() && gate->defined()) {
        CHECK_CUDA_F32((*gate));
        TORCH_CHECK(gate->is_contiguous() && gate->numel() == x.numel(), "conv_cast_bf16: gate shape");
        g = gate->data_ptr<float>();
    }
    if ((reinterpret_cast<uintptr_t>(x.data_ptr<float>()) & 15) || (reinterpret_cast<uintptr_t>(g) & 15))   // 128-bit loads need 16-byte bases
        return g ? (x * gate->gt(0).view_as(x)).to(torch::kBFloat16) : x.to(torch::kBFloat16);
    auto out = torch::empty(x.sizes(), x.options().dtype(torch::kBFloat16));
    CHECK_OK(fdb::conv_cast_bf16_launch(x.data_ptr<float>(), g, out.data_ptr(), x.numel(), cur_stream()), "conv_cast_bf16");
    return out;
}
// strided rows [n, numel] fp32 (stride(1) == 1; the staged parameter rows of the stacked pairs) -> contiguous bf16 [n, numel]
Tensor conv_cast_rows_bf16(Tensor x) {
    CHECK_CUDA_F32(x);
    TORCH_CHECK(x.dim() == 2 && x.stride(1) == 1 && x.size(1) % 8 == 0 && x.stride(0) % 4 == 0 &&
                (reinterpret_cast<uintptr_t>(x.data_ptr<float>()) & 15) == 0, "conv_cast_rows_bf16: [n, numel] rows, 16-byte aligned, numel % 8 == 0");
    c10::cuda::CUDAGuard guard(x.device());
    auto out = torch::empty({x.size(0), x.size(1)}, x.options().dtype(torch::kBFloat16));
    CHECK_OK(fdb::conv_cast_rows_bf16_launch(x.data_ptr<float>(), x.stride(0), out.data_ptr(), (int)x.size(0), x.size(1), cur_stream()), "conv_cast_rows_bf16");
    return out;
}
// xb: bf16 NHWC [N, H, W, G·C]; wq: bf16 [G·Cout][R][S][C]; -> fp32 NHWC [N, P, Q, G·Cout] = act(conv(x, w) + bias), G groups
Tensor conv_tma_fwd(Tensor xb, Tensor wq, c10::optional<Tensor> bias, int64_t stride, int64_t pad, bool relu, int64_t groups) {
    TORCH_CHECK(xb.is_cuda() && xb.scalar_type() == torch::kBFloat16 && xb.dim() == 4 && xb.is_contiguous(), "conv_tma_fwd: xb must be contiguous bf16 NHWC");
    TORCH_CHECK(wq.is_cuda() && wq.scalar_type() == torch::kBFloat16 && wq.dim() == 4 && wq.is_contiguous(), "conv_tma_fwd: wq must be bf16 [K,R,S,C]");
    const int G = (int)groups;
    const int N = (int)xb.size(0), H = (int)xb.size(1), W = (int)xb.size(2), C = (int)wq.size(3);
    const int R = (int)wq.size(1), S = (int)wq.size(2);
    TORCH_CHECK(G >= 1 && wq.size(0) % G == 0 && xb.size(3) == (int64_t)G * C, "conv_tma_fwd: group shapes");
    const int K = (int)(wq.size(0) / G);
    TORCH_CHECK(C % 64 == 0 && K % 8 == 0 && R == S && (G == 1 || K % 32 == 0), "conv_tma_fwd: needs Cin % 64 == 0, Cout % 8 == 0 (% 32 grouped), square filter");
    const int P = (H + 2 * (int)pad - R) / (int)stride + 1, Q = (W + 2 * (int)pad - S) / (int)stride + 1;
    TORCH_CHECK(P > 0 && Q > 0 && pad >= 0 && pad < 128 && stride >= 1 && stride <= 8, "conv_tma_fwd: geometry");
    c10::cuda::CUDAGuard guard(xb.device());
    auto y = torch::empty({N, P, Q, (int64_t)G * K}, xb.options().dtype(torch::kFloat32));
    Tensor bias_f;
    const float* bp = nullptr;
    if (bias.has_value() && bias->defined()) {
        bias_f = bias->to(torch::kFloat32).contiguous();
        TORCH_CHECK(bias_f.numel() == (int64_t)G * K, "conv_tma_fwd: bias size");
        bp = bias_f.data_ptr<float>();
    }
    CHECK_OK(fdb::conv_tma_fwd_launch(xb.data_ptr(), wq.data_ptr(), y.data_ptr<float>(), bp, N, H, W, C, K, R, S, P, Q, (int)pad, (int)stride,
                                      0, relu ? 1 : 0, G, cur_stream()), "conv_tma_fwd (tcgen05 + TMA im2col)");
    return y;
}
// stride-1 data gradient.  dyb: bf16 NHWC [N, P, Q, G·Cout]; wq: THE FORWARD pack bf16 [G·Cout][R][S][Cin] (read as an MN-major operand
// with flipped taps); pad = the forward padding; -> dx fp32 NHWC [N, P + R - 1 - 2·pad, Q + S - 1 - 2·pad, G·Cin]
Tensor conv_tma_dgrad(Tensor dyb, Tensor wq, int64_t pad, int64_t groups) {
    TORCH_CHECK(dyb.is_cuda() && dyb.scalar_type() == torch::kBFloat16 && dyb.dim() == 4 && dyb.is_contiguous(), "conv_tma_dgrad: dyb must be contiguous bf16 NHWC");
    TORCH_CHECK(wq.is_cuda() && wq.scalar_type() == torch::kBFloat16 && wq.dim() == 4 && wq.is_contiguous(), "conv_tma_dgrad: wq must be bf16 [K,R,S,C]");
    const int G = (int)groups;
    const int N = (int)dyb.size(0), P = (int)dyb.size(1), Q = (int)dyb.size(2);
    const int R = (int)wq.size(1), S = (int)wq.size(2), C = (int)wq.size(3);
    TORCH_CHECK(G >= 1 && wq.size(0) % G == 0 && dyb.size(3) == wq.size(0), "conv_tma_dgrad: group shapes");
    const int K = (int)(wq.size(0) / G);
    TORCH_CHECK(K % 64 == 0 && C % 8 == 0 && R == S && pad >= 0 && pad <= R - 1 && (G == 1 || C % 32 == 0),
                "conv_tma_dgrad: needs Cout % 64 == 0, Cin % 8 == 0 (% 32 grouped), square filter, pad <= R-1");
    const int pd = R - 1 - (int)pad, H = P + 2 * pd - R + 1, W = Q + 2 * pd - S + 1;
    c10::cuda::CUDAGuard guard(dyb.device());
    auto dx = torch::empty({N, H, W, (int64_t)G * C}, dyb.options().dtype(torch::kFloat32));
    CHECK_OK(fdb::conv_tma_fwd_launch(dyb.data_ptr(), wq.data_ptr(), dx.data_ptr<float>(), nullptr, N, P, Q, K, C, R, S, H, W, pd, 1, 1, 0, G,
                                      cur_stream()), "conv_tma_dgrad (tcgen05 + TMA im2col)");
    return dx;
}
// xb: bf16 NHWC [N, H, W, G·C]; dyb: bf16 NHWC [N, P, Q, G·K]; dw: fp32 — [K, R, S, C] contiguous (G = 1) or rows [G, K·R·S·C] with
// stride(1) == 1 and any 16-byte-multiple row stride (the flat gradient rows of the stacked pairs); the gradient is ADDED into it
void conv_tma_wgrad(Tensor xb, Tensor dyb, Tensor dw, int64_t R, int64_t stride, int64_t pad, int64_t groups) {
    TORCH_CHECK(xb.is_cuda() && xb.scalar_type() == torch::kBFloat16 && xb.dim() == 4 && xb.is_contiguous(), "conv_tma_wgrad: xb must be contiguous bf16 NHWC");
    TORCH_CHECK(dyb.is_cuda() && dyb.scalar_type() == torch::kBFloat16 && dyb.dim() == 4 && dyb.is_contiguous(), "conv_tma_wgrad: dyb must be contiguous bf16 NHWC");
    CHECK_CUDA_F32(dw);
    const int G = (int)groups;
    TORCH_CHECK(G >= 1 && xb.size(3) % G == 0 && dyb.size(3) % G == 0 && dyb.size(0) == xb.size(0), "conv_tma_wgrad: group shapes");
    const int N = (int)xb.size(0), H = (int)xb.size(1), W = (int)xb.size(2), C = (int)(xb.size(3) / G);
    const int P = (int)dyb.size(1), Q = (int)dyb.size(2), K = (int)(dyb.size(3) / G);
    const int64_t numel = (int64_t)K * R * R * C;
    long long gstride = numel;
    if (G == 1) {
        TORCH_CHECK(dw.is_contiguous() && dw.numel() == numel, "conv_tma_wgrad: dw must be a contiguous fp32 [K,R,S,C] buffer");
    } else {
        TORCH_CHECK(dw.dim() == 2 && dw.size(0) == G && dw.size(1) == numel && dw.stride(1) == 1, "conv_tma_wgrad: dw must be rows [G, K·R·S·C]");
        gstride = dw.stride(0);
    }
    TORCH_CHECK(C % 64 == 0 && K % 8 == 0, "conv_tma_wgrad: needs Cin % 64 == 0, Cout % 8 == 0");
    c10::cuda::CUDAGuard guard(xb.device());
    CHECK_OK(fdb::conv_tma_wgrad_launch(xb.data_ptr(), dyb.data_ptr(), dw.data_ptr<float>(), N, H, W, C, K, (int)R, (int)R, P, Q, (int)pad,
                                        (int)stride, G, gstride, cur_stream()), "conv_tma_wgrad (tcgen05 + TMA im2col)");
}
// bf16 [K][R][S][C] (the cast channels_last weight) -> bf16 [C][R][S][K] for the software-gather data-gradient kernel
Tensor conv_pack_t(Tensor wq) {
    TORCH_CHECK(wq.is_cuda() && wq.scalar_type() == torch::kBFloat16 && wq.dim() == 4 && wq.is_contiguous(), "conv_pack_t: wq must be bf16 [K,R,S,C]");
    c10::cuda::CUDAGuard guard(wq.device());
    const int K = (int)wq.size(0), R = (int)wq.size(1), S = (int)wq.size(2), C = (int)wq.size(3);
    auto out = torch::empty({C, R, S, K}, wq.options());
    CHECK_OK(fdb::conv_pack_t_launch(wq.data_ptr(), out.data_ptr(), K, C, R * S, cur_stream()), "conv_pack_t");
    return out;
}

// bias / W_ih1 / embedding gradients of every chunk from the gate-gradient histories (lstm_tc.cu::lstm_small_grads_kernel)
std::vector<Tensor> lstm_small_grads(Tensor params, Tensor row_off, int64_t off_emb, int64_t off_wih1, Tensor tokens, Tensor dgates,
                                     int64_t E, int64_t V) {
    CHECK_CUDA_F32(params); CHECK_CUDA_I32(tokens);
    TORCH_CHECK(row_off.is_cuda() && row_off.scalar_type() == torch::kInt64, "row_off must be a CUDA int64 tensor");
    TORCH_CHECK(dgates.is_cuda() && dgates.scalar_type() == torch::kBFloat16 && dgates.is_contiguous(), "dgates must be CUDA bf16");
    c10::cuda::CUDAGuard guard(params.device());
    const int64_t n = tokens.size(0), T = tokens.size(2);
    TORCH_CHECK(row_off.numel() == n && dgates.numel() == 2 * n * T * 16 * 1024, "lstm_small_grads: sizes");
    auto o = params.options();
    auto db1 = torch::empty({n, 1024}, o), db2 = torch::empty({n, 1024}, o), dw = torch::empty({n, 1024, E}, o);
    auto de = torch::empty({n, 8, V, E}, o);
    fdb::LstmSmallArgs a{};
    a.params = params.data_ptr<float>();
    a.row_off = reinterpret_cast<const long long*>(row_off.data_ptr<int64_t>());
    a.off_emb = off_emb; a.off_wih1 = off_wih1;
    a.tokens = tokens.data_ptr<int>(); a.dgates = dgates.data_ptr();
    a.db1 = db1.data_ptr<float>(); a.db2 = db2.data_ptr<float>(); a.dwih1 = dw.data_ptr<float>(); a.demb_part = de.data_ptr<float>();
    a.T = (int)T; a.E = (int)E; a.V = (int)V;
    CHECK_OK(fdb::lstm_small_grads_launch(a, (int)n, cur_stream()), "lstm_small_grads");
    return {db1, db2, dw, de.sum(1)};
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    namespace py = pybind11;
    m.def("fed_round_small", &fed_round_small, py::arg("kind"), py::arg("din"), py::arg("hid"), py::arg("dout"), py::arg("X"),
          py::arg("Y"), py::arg("nsamp"), py::arg("W"), py::arg("theta"), py::arg("theta_stride"), py::arg("opt_m"), py::arg("opt_v"),
          py::arg("opt_vmax"), py::arg("opt_step"), py::arg("train_index"), py::arg("train_count"), py::arg("feat_mask"),
          py::arg("eval_train_model"), py::arg("eval_test_model"), py::arg("ens_w"), py::arg("client_out"), py::arg("lr_dev"),
          py::arg("metrics"), py::arg("timers"), py::arg("fcfg"), py::arg("icfg"), py::arg("peer_inbox"), py::arg("error_flag"),
          py::arg("counters"), py::arg("peer_metrics"), py::arg("host_io"), py::arg("participants") = py::none());
    m.def("fed_round_small_supported", &fed_round_small_supported);
    m.def("fed_round_small_fits", &fed_round_small_fits);
    m.def("fed_round_small_launch_shape", &fed_round_small_launch_shape);
    m.def("mlp_eval_matrix", &mlp_eval_matrix);
    m.def("cluster_aggregate", &cluster_aggregate);
    m.def("cluster_aggregate_opt", &cluster_aggregate_opt);
    m.def("weighted_average", &weighted_average);
    m.def("fedavg_reduce_apply_peer", &fedavg_reduce_apply_peer);
    m.def("merge_axpby", &merge_axpby);
    m.def("mean_sq_diff", &mean_sq_diff);
    m.def("gossip_mix", &gossip_mix);
    m.def("robust_clip", &robust_clip);
    m.def("eval_logits", &eval_logits);
    m.def("aue_sqerr", &aue_sqerr);
    m.def("ensemble_vote", &ensemble_vote);
    m.def("confusion_matrix", &confusion_matrix);
    m.def("adam_amsgrad_rows", &adam_amsgrad_rows);
    m.def("sgd_rows", &sgd_rows);
    m.def("gram_cosine", &gram_cosine);
    m.def("modp_matmul", &modp_matmul);
    m.def("kd_kl_fwd_bwd", &kd_kl_fwd_bwd);
    m.def("vfl_bce_grad", &vfl_bce_grad);
    m.def("group_norm_fwd", &group_norm_fwd);
    m.def("group_norm_fwd_train", &group_norm_fwd_train);
    m.def("group_norm_bwd", &group_norm_bwd);
    m.def("bn_nhwc_fwd", &bn_nhwc_fwd);
    m.def("bn_nhwc_bwd", &bn_nhwc_bwd);
    m.def("gemm_tn_bias_act", &gemm_tn_bias_act);
    m.def("gemm_tn_bias_act_peer", &gemm_tn_bias_act_peer);
    m.def("gemm_bias_act", &gemm_bias_act);
    m.def("gemm_batched_mn", &gemm_batched_mn);
    m.def("gossip_mix_peer", &gossip_mix_peer);
    m.def("graph_launch_sync", &graph_launch_sync);
    m.def("im2col_bf16", &im2col_bf16);
    m.def("col2im", &col2im);
    m.def("lstm2_forward", &lstm2_forward);
    m.def("lstm2_backward", &lstm2_backward);
    m.def("lstm_head", &lstm_head);
    m.def("lstm_small_grads", &lstm_small_grads);
    m.def("conv_igemm_fwd", &conv_igemm_fwd);
    m.def("conv_cast_bf16", &conv_cast_bf16);
    m.def("conv_tma_fwd", &conv_tma_fwd);
    m.def("conv_tma_wgrad", &conv_tma_wgrad);
    m.def("conv_tma_dgrad", &conv_tma_dgrad);
    m.def("conv_cast_rows_bf16", &conv_cast_rows_bf16);
    m.def("gemm_debug_counters", []() {
        std::vector<int64_t> v(16);
        cudaDeviceSynchronize();
        CHECK_OK(fdb::gemm_debug_counters(reinterpret_cast<long long*>(v.data())), "gemm_debug_counters");
        return v;
    });
    m.def("conv_pack_t", &conv_pack_t);
    m.def("conv_igemm_dgrad", &conv_igemm_dgrad);
    m.def("conv_igemm_wgrad", &conv_igemm_wgrad);
}
