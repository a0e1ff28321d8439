// fed_round_small — one persistent kernel runs R complete federated rounds of a small-MLP federation:
//
//   broadcast (cluster models are smem-resident)  →  E local optimizer steps for every active
//   (client, model) pair, one warp per pair, parameters + gradients in registers  →  per-cluster weighted
//   FedAvg aggregation (warp → CTA smem → thread-block-cluster DSMEM → [multi-GPU] NVLink peer inboxes)
//   →  optional IFCA re-clustering  →  train/test evaluation of every client (optionally ensemble vote)
//
// with no host involvement between rounds.  This is K3(a)+K1+K2+K4 of SURVEY §2.9 fused; it replaces, per
// round, N pickled sends of M state_dicts, N·M load_state_dict, 5·N·M_active eager optimizer steps
// (~10 launches each), N pickled uploads, a python for-key-for-client average and 2N eager evaluations with
// per-batch .item() syncs (reference: FedAvgEnsServerManager.py:36-67, FedAvgEnsTrainerSoftCluster.py:63-135,
// FedAvgEnsAggregatorSoftCluster.py:137-285).
//
// Work decomposition (SEA fnn: P = 38 parameters, B ≤ 500 samples per batch):
//   * one WARP per (client, model) pair; lanes split the mini-batch; every lane keeps θ (P regs) and its
//     partial gradient (P regs) in registers; the P×32 partials are transposed through padded smem so lane l
//     owns column sums / optimizer state of parameters l, l+32, … (bank-conflict free both ways);
//   * pairs are compacted per round from the device-resident weight tensor W[t',m,c] (membership is data —
//     no re-capture / re-launch when clustering changes) and dealt round-robin to the warps of a
//     thread-block CLUSTER; partial sums meet through distributed shared memory with ONE cluster barrier
//     per round (double-buffered partials);
//   * multi-GPU: each rank owns clients c ≡ rank (mod world); after the cluster reduction CTA 0 pushes the
//     M×P partial to every peer's symmetric inbox with plain st.global over NVLink, publishes a
//     st.release.sys epoch flag, and every CTA acquires the world's flags and sums the inbox in rank order
//     (bit-identical on all ranks, no NCCL, one one-way NVLink latency per round).
#include <cooperative_groups.h>

#include "fed_round_small.h"
#include "mlp.cuh"

namespace cg = cooperative_groups;

namespace fdb {

template <class Net>
struct SmallCfg {
    static constexpr int P = Net::P;
    static constexpr int kThreads = (P <= 24) ? 512 : (P <= 40 ? 384 : 256);  // register budget ≈ 2P + 90 live values
    static constexpr int kWarps = kThreads / 32;
    static constexpr int kCols = (P + 31) / 32;  // parameters owned per lane
};

constexpr int kTmax = 64;  // the fused kernel supports t_cur < kTmax time steps (host falls back otherwise)

struct SmemLayout {
    int theta, part, slot, slot_model, gbuf, thl, wsum, ptab_nb, ptab_w, ncm, tot, active, pairs, misc, total;
};

template <class Net>
__host__ __device__ inline SmemLayout make_layout(int M, int C, int pairs_per_cta) {
    using Cfg = SmallCfg<Net>;
    constexpr int P = Net::P;
    SmemLayout L;
    int o = 0;
    auto take = [&](int nfloats) { int r = o; o += (nfloats + 3) & ~3; return r; };
    L.theta = take(M * P);
    L.part = take(2 * M * P);
    L.slot = take(pairs_per_cta * P);
    L.slot_model = take(pairs_per_cta);
    L.gbuf = take(Cfg::kWarps * P * 33);
    L.thl = take(Cfg::kWarps * P);
    L.wsum = take(Cfg::kWarps * P);
    L.ptab_nb = take(Cfg::kWarps * kTmax);
    L.ptab_w = take(Cfg::kWarps * kTmax);
    L.ncm = take(C * M);
    L.tot = take(M);
    L.active = take(M);
    L.pairs = take(C * M);
    L.misc = take(8);
    L.total = o;
    return L;
}

// barrier among the WPP warps of a pair group (named barrier 1 + group id; id 0 is __syncthreads)
FDB_DEVICE void group_barrier(int wpp, int gidx) {
    if (wpp == 1) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(1 + gidx), "r"(wpp * 32) : "memory");
}

// sample coordinates of element i of the current mini-batch
struct BatchSel {
    int mode;        // 0/1: contiguous [lo, lo+n) of (tb, c);  2: list
    int tb, lo, n;
    const int* list; // mode 2: flat sample ids
};

// kPart: a participants table is present (partial participation); the full-participation instance carries none of its code
template <class Net, bool kPart>
__global__ void __launch_bounds__(SmallCfg<Net>::kThreads, 1) fed_round_small_kernel(const __grid_constant__ RoundParams p) {
    using Cfg = SmallCfg<Net>;
    constexpr int P = Net::P, IN = Net::kIn, OUT = Net::kOut, HID = Net::kHid;
    constexpr int NW = Cfg::kWarps, COLS = Cfg::kCols;
    extern __shared__ __align__(16) float smem[];

    cg::cluster_group cluster = cg::this_cluster();
    const int G = (int)cluster.num_blocks();
    const int crank = (int)cluster.block_rank();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int C = p.C, M = p.M, S = p.S, t = p.t_cur, B = p.batch_size;
    const int CM = C * M, MP = M * P;
    const int pairs_per_cta = ((kPart ? p.K : C) * M + G - 1) / G;   // must match launch_shape on the host
    const SmemLayout L = make_layout<Net>(M, C, pairs_per_cta);
    float* theta_s = smem + L.theta;
    float* part_s = smem + L.part;
    float* slot_s = smem + L.slot;
    int* slot_model = reinterpret_cast<int*>(smem + L.slot_model);
    const int WPP = (p.warps_per_pair == 4 || p.warps_per_pair == 2) ? p.warps_per_pair : 1;
    const int NG = NW / WPP;                    // pair groups per CTA
    const int gidx = warp / WPP, sub = warp % WPP;
    float* gbuf = smem + L.gbuf + warp * (P * 33);
    float* thl = smem + L.thl + gidx * P;                    // group-local model
    float* wsum = smem + L.wsum + gidx * (WPP * P);          // per-warp column sums of the group
    int* ptab_nb = reinterpret_cast<int*>(smem + L.ptab_nb) + gidx * kTmax;
    float* ptab_w = smem + L.ptab_w + gidx * kTmax;
    float* ncm_s = smem + L.ncm;
    float* tot_s = smem + L.tot;
    int* active_s = reinterpret_cast<int*>(smem + L.active);
    int* pairs_s = reinterpret_cast<int*>(smem + L.pairs);
    int* misc_s = reinterpret_cast<int*>(smem + L.misc);  // [0] = npairs

    if (p.host_x != nullptr) {
        // ---- fused H2D: this round's inputs come straight from pinned host memory (each CTA copies 1/G of the range)
        const size_t gthreads = (size_t)G * blockDim.x, gt = (size_t)crank * blockDim.x + tid;
        const size_t xoff = (size_t)p.host_t0 * C * S * IN, xn = (size_t)p.host_steps * C * S * IN;
        const size_t yoff = (size_t)p.host_t0 * C * S, yn = (size_t)p.host_steps * C * S;
        float* Xd = const_cast<float*>(p.X) + xoff;
        int* Yd = const_cast<int*>(p.Y) + yoff;
        if (((xoff | xn) & 3) == 0) {
            for (size_t i = gt; i < xn / 4; i += gthreads) {
                float4 v;
                asm volatile("ld.global.relaxed.sys.v4.f32 {%0, %1, %2, %3}, [%4];"
                             : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p.host_x + 4 * i) : "memory");
                reinterpret_cast<float4*>(Xd)[i] = v;
            }
        } else {
            for (size_t i = gt; i < xn; i += gthreads) Xd[i] = ld_relaxed_sys_f32(p.host_x + i);
        }
        if (((yoff | yn) & 3) == 0) {
            for (size_t i = gt; i < yn / 4; i += gthreads) {
                int4 v;
                asm volatile("ld.global.relaxed.sys.v4.s32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p.host_y + 4 * i) : "memory");
                reinterpret_cast<int4*>(Yd)[i] = v;
            }
        } else {
            for (size_t i = gt; i < yn; i += gthreads) Yd[i] = __float_as_int(ld_relaxed_sys_f32(reinterpret_cast<const float*>(p.host_y) + i));
        }
        __threadfence();
        if (G > 1) cluster.sync(); else __syncthreads();   // every CTA sees the whole copied range
    }
    // ---- cold-start: pull the (remaining) working set — samples of the steps that were not just copied in — into L2
    //      with one wave of prefetches
    {
        const int steps = p.host_x ? min(p.host_t0, p.T1) : min(t + 2, p.T1);
        const size_t xb = (size_t)steps * C * S * IN * sizeof(float), yb = (size_t)steps * C * S * sizeof(int);
        const size_t gthreads = (size_t)G * blockDim.x, gt = (size_t)crank * blockDim.x + tid;
        for (size_t off = gt * 128; off < xb; off += gthreads * 128)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.X) + off));
        for (size_t off = gt * 128; off < yb; off += gthreads * 128)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.Y) + off));
        // optimizer moments / step counters / plan tables: small, but every pair's first touch would be a DRAM miss
        const size_t ob = (size_t)CM * P * sizeof(float);
        if (p.use_adam && p.opt_m)
            for (size_t off = gt * 128; off < ob; off += gthreads * 128) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.opt_m) + off));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.opt_v) + off));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.opt_vmax) + off));
            }
        const size_t wb = (size_t)(t + 1) * CM * sizeof(float);
        for (size_t off = gt * 128; off < wb; off += gthreads * 128)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.W) + off));
        if (gt * 128 < (size_t)CM * sizeof(int)) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.opt_step) + gt * 128));
        if (gt * 128 < (size_t)p.T1 * C * sizeof(int)) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.nsamp) + gt * 128));
    }
    // ---- load the cluster models once (broadcast == this smem fill; afterwards θ never leaves the SM) ----
    for (int e = tid; e < MP; e += blockDim.x) theta_s[e] = p.theta[(e / P) * p.theta_stride + (e % P)];
    const float lr = p.lr_ptr ? *p.lr_ptr : p.lr;
    // graph-replay friendly: the round number (RNG stream) and the cross-GPU epoch come from device counters
    const int round0 = p.counters ? p.counters[0] : p.round0;
    const unsigned flag_base = p.counters ? (unsigned)p.counters[1] : p.flag_base;
    const float b1 = p.beta1, b2 = p.beta2;
    bool need_prep = true;
    __syncthreads();

    for (int r = 0; r < p.rounds; ++r) {
        const unsigned rnd = (unsigned)(round0 + r);
        const int buf = r & 1;

        // ------------------------------------------------------------------ prep: pair list from W
        if (need_prep) {
            // partial participation: this round's worker slots → client ids (slot s trains client prow[s]); the table has
            // one row per round of the time step, rounds past its end wrap around
            const int* prow = kPart ? p.participants + (size_t)((round0 + r) % p.part_rows) * p.K : nullptr;
            const int nslots = prow ? p.K : C;
            for (int k = tid; k < CM; k += blockDim.x) {
                const int c = k / M, m = k % M;
                float n = 0.f;
                if (p.sample_mode == 2) {
                    n = (float)p.train_count[m * C + c];
                } else if (p.sample_mode == 1) {
                    float wsum = 0.f; int nbsum = 0;
                    for (int tt = 0; tt <= t; ++tt) {
                        wsum += p.W[(tt * M + m) * C + c];
                        nbsum += (p.nsamp[tt * C + c] + B - 1) / B;
                    }
                    n = (wsum > 0.f) ? (float)nbsum : 0.f;
                } else {
                    float nbw = 0.f, nsw = 0.f;
                    for (int tt = 0; tt <= t; ++tt) {
                        const float w = p.W[(tt * M + m) * C + c];
                        const int ns = p.nsamp[tt * C + c];
                        nbw += w * (float)((ns + B - 1) / B);
                        nsw += w * (float)ns;
                    }
                    n = (nbw > 0.f) ? (p.n_mode == 1 ? nsw : nbw) : 0.f;
                }
                ncm_s[k] = n;
            }
            __syncthreads();
            for (int m = tid; m < M; m += blockDim.x) {
                int act = 0;
                if (p.sample_mode == 2) {
                    for (int c = 0; c < C; ++c) act |= (p.train_count[m * C + c] > 0);
                } else {
                    for (int c = 0; c < C; ++c) act |= (p.W[(t * M + m) * C + c] != 0.f);
                }
                float tot = 0.f;   // aggregation weight total over the clients that train this round
                if (act) for (int s = 0; s < nslots; ++s) tot += ncm_s[(prow ? prow[s] : s) * M + m];
                active_s[m] = act;
                tot_s[m] = tot;
            }
            __syncthreads();
            if (warp == 0) {  // ordered stream compaction of participating, locally-owned pairs; keys are slot-major s·M + m
                int base = 0;
                const int SM = nslots * M;
                for (int k0 = 0; k0 < SM; k0 += 32) {
                    const int k = k0 + lane;
                    bool on = false;
                    int c = 0;
                    if (k < SM) {
                        const int s = k / M, m = k % M;
                        c = prow ? prow[s] : s;
                        on = active_s[m] && ncm_s[c * M + m] > 0.f && (p.world == 1 || (c % p.world) == p.rank);
                    }
                    const unsigned mask = __ballot_sync(0xffffffffu, on);
                    // with a table: entry = client << 16 | key (C·M < 2^16: ncm and the pair list alone must fit in 227 KB of
                    // shared memory)
                    if (on) pairs_s[base + __popc(mask & ((1u << lane) - 1u))] = kPart ? ((c << 16) | k) : k;
                    base += __popc(mask);
                }
                if (lane == 0) misc_s[0] = base;
            }
            __syncthreads();
            need_prep = (p.recluster_hard != 0) || kPart;
        }
        const int npairs = misc_s[0];

        // ------------------------------------------------------------------ local training: WPP warps per pair
        // A *group* of WPP warps (1, 2 or 4) owns one (client, model) pair: the mini-batch is strided over the
        // group's lanes; every warp transposes its lanes' partial gradients through padded smem so lane l holds the
        // column sums of parameters l, l+32, …; the group's leader warp adds the WPP partial columns, applies the
        // optimizer for the columns it owns and publishes the new local model; two named barriers per step.
        if (gidx < NG) {
        for (int i = crank + G * gidx; i < npairs; i += G * NG) {
            const int e = pairs_s[i];
            const int k = kPart ? (e & 0xFFFF) : e;       // slot-major: optimizer state / client_out row of worker slot k / M
            const int c = kPart ? (e >> 16) : k / M;      // the client that slot trains this round (data, batch hash)
            const int m = k % M;
            const int li = i / G;
            float th[P];
#pragma unroll
            for (int q = 0; q < P; ++q) th[q] = theta_s[m * P + q];
            float om[COLS], ov[COLS], ovm[COLS];
            int ostep = 0;
            const size_t obase = (size_t)k * P;
            double b1pow = 1.0, b2pow = 1.0;
            if (sub == 0) {
#pragma unroll
                for (int q = 0; q < COLS; ++q)  // thl = the group's local model; leader lane l owns entries l, l+32, …
                    if (lane + 32 * q < P) thl[lane + 32 * q] = theta_s[m * P + lane + 32 * q];
                if (p.use_adam) {
                    ostep = p.opt_step[k];
#pragma unroll
                    for (int q = 0; q < COLS; ++q) {
                        const int pp = lane + 32 * q;
                        om[q] = pp < P ? p.opt_m[obase + pp] : 0.f;
                        ov[q] = pp < P ? p.opt_v[obase + pp] : 0.f;
                        ovm[q] = pp < P ? p.opt_vmax[obase + pp] : 0.f;
                    }
                    if (ostep > 0) { b1pow = pow((double)b1, (double)ostep); b2pow = pow((double)b2, (double)ostep); }
                }
                // per-pair batch-pool table (t_cur < kTmax is enforced on the host)
                for (int tt = lane; tt <= t; tt += 32) {
                    const int nb = (p.nsamp[tt * C + c] + B - 1) / B;
                    const float w = (p.sample_mode == 2) ? 0.f : p.W[(tt * M + m) * C + c];
                    ptab_nb[tt] = (p.sample_mode == 0) ? ((w * (float)nb > 0.f) ? nb : 0) : nb;
                    ptab_w[tt] = w;
                }
            }
            float fm[IN];
#pragma unroll
            for (int q = 0; q < IN; ++q) fm[q] = p.feat_mask ? p.feat_mask[m * IN + q] : 1.f;
            group_barrier(WPP, gidx);
            int npool = 0; float wtot = 0.f;
            if (p.sample_mode == 0) { for (int tt = 0; tt <= t; ++tt) npool += ptab_nb[tt]; }
            else if (p.sample_mode == 1) { for (int tt = 0; tt <= t; ++tt) wtot += ptab_w[tt]; }
            const int cnt = (p.sample_mode == 2) ? p.train_count[m * C + c] : 0;
            const int* list = (p.sample_mode == 2) ? p.train_index + (size_t)(m * C + c) * p.Lmax : nullptr;

            for (int step = 0; step < p.epochs; ++step) {
                const unsigned h1 = batch_hash(p.seed, rnd, (unsigned)c, (unsigned)m, (unsigned)step);
                int sel_tb = 0, sel_lo = 0, sel_n = 0;
                if (p.sample_mode == 0) {
                    int j = (int)hash_choice(h1, (unsigned)npool);
                    for (int tt = 0; tt <= t; ++tt) {
                        const int nb = ptab_nb[tt];
                        if (j < nb) { sel_tb = tt; sel_lo = j * B; sel_n = min(B, p.nsamp[tt * C + c] - j * B); break; }
                        j -= nb;
                    }
                } else if (p.sample_mode == 1) {
                    const unsigned h2 = mix32(h1 ^ 0x68E31DA4u);
                    const float u = __uint2float_rn(h1 >> 8) * 5.9604644775390625e-8f * wtot;
                    float cum = 0.f; int tt_sel = 0;
                    for (int tt = 0; tt <= t; ++tt) { cum += ptab_w[tt]; if (cum <= u) tt_sel = tt + 1; }
                    tt_sel = min(tt_sel, t);
                    while (tt_sel > 0 && ptab_nb[tt_sel] == 0) --tt_sel;
                    const int ns = p.nsamp[tt_sel * C + c];
                    const int b = (int)hash_choice(h2, (unsigned)max(ptab_nb[tt_sel], 1));
                    sel_tb = tt_sel; sel_lo = b * B; sel_n = max(min(B, ns - b * B), 0);
                } else {
                    const int nbm = (cnt + B - 1) / B;
                    const int b = (int)hash_choice(h1, (unsigned)nbm);
                    sel_lo = b * B; sel_n = min(B, cnt - b * B);
                }
                float g[P];
#pragma unroll
                for (int q = 0; q < P; ++q) g[q] = 0.f;
                const float scale = 1.0f / (float)max(sel_n, 1);
                for (int sidx = sub * 32 + lane; sidx < sel_n; sidx += 32 * WPP) {
                    int tb = sel_tb, sx = sel_lo + sidx;
                    if (p.sample_mode == 2) { const int qid = list[sel_lo + sidx]; tb = qid / S; sx = qid - tb * S; }
                    const size_t row = (size_t)(tb * C + c) * S + sx;
                    float x[IN];
#pragma unroll
                    for (int q = 0; q < IN; ++q) x[q] = p.X[row * IN + q] * fm[q];
                    const int y = p.Y[row];
                    float z[OUT], h[HID > 0 ? HID : 1], pr[OUT];
                    int am;
                    Net::forward(th, x, z, h);
                    Net::softmax_ce(z, y, pr, am);
                    Net::backward_accum(th, x, z, h, pr, y, scale, g);
                }
                // transpose-reduce inside the warp: lane l ends up with Σ_lanes g[p] for p = l + 32q
#pragma unroll
                for (int q = 0; q < P; ++q) gbuf[q * 33 + lane] = g[q];
                __syncwarp();
                float gcol[COLS];
#pragma unroll
                for (int q = 0; q < COLS; ++q) {
                    const int pp = lane + 32 * q;
                    float gs = 0.f;
                    if (pp < P) {
#pragma unroll 8
                        for (int j = 0; j < 32; ++j) gs += gbuf[pp * 33 + j];
                        if (WPP > 1) wsum[sub * P + pp] = gs;
                    }
                    gcol[q] = gs;
                }
                if (WPP > 1) group_barrier(WPP, gidx);
                if (sub == 0) {
                    float step_size = lr, bc2_sqrt = 1.f;
                    if (p.use_adam) {  // bias corrections from running fp64 powers; the divisions/sqrt run in fp32
                        ++ostep;
                        b1pow *= (double)b1;
                        b2pow *= (double)b2;
                        step_size = lr / (float)(1.0 - b1pow);
                        bc2_sqrt = sqrtf((float)(1.0 - b2pow));
                    }
#pragma unroll
                    for (int q = 0; q < COLS; ++q) {
                        const int pp = lane + 32 * q;
                        if (pp < P) {
                            float gs = gcol[q];
                            for (int w2 = 1; w2 < WPP; ++w2) gs += wsum[w2 * P + pp];
                            float w = thl[pp];
                            if (p.use_adam) {
                                gs = fmaf(p.wd, w, gs);
                                om[q] = fmaf(gs - om[q], 1.0f - b1, om[q]);
                                ov[q] = fmaf((1.0f - b2) * gs, gs, ov[q] * b2);
                                ovm[q] = fmaxf(ovm[q], ov[q]);
                                const float denom = sqrtf(ovm[q]) / bc2_sqrt + p.eps;
                                w = w - step_size * (om[q] / denom);
                            } else {
                                w = w - lr * gs;
                            }
                            thl[pp] = w;
                        }
                    }
                }
                group_barrier(WPP, gidx);
#pragma unroll
                for (int q = 0; q < P; ++q) th[q] = thl[q];
            }
            if (sub == 0) {  // persist optimizer state, publish the weighted local model
                if (p.use_adam) {
#pragma unroll
                    for (int q = 0; q < COLS; ++q) {
                        const int pp = lane + 32 * q;
                        if (pp < P) { p.opt_m[obase + pp] = om[q]; p.opt_v[obase + pp] = ov[q]; p.opt_vmax[obase + pp] = ovm[q]; }
                    }
                    if (lane == 0) p.opt_step[k] = ostep;
                }
                const float wgt = ncm_s[kPart ? c * M + m : k] / tot_s[m];
#pragma unroll
                for (int q = 0; q < COLS; ++q) {
                    const int pp = lane + 32 * q;
                    if (pp < P) {
                        slot_s[li * P + pp] = thl[pp] * wgt;
                        if (p.client_out && r == p.rounds - 1) p.client_out[obase + pp] = thl[pp];
                    }
                }
                if (lane == 0) slot_model[li] = m;
            }
            group_barrier(WPP, gidx);  // thl / ptab are rewritten by the next pair
        }
        }
        __syncthreads();
        if (p.timers && crank == 0 && blockIdx.x == 0 && tid == 0) p.timers[r * 4 + 0] = globaltimer_ns();

        // ------------------------------------------------------------------ aggregation
        if (!p.skip_aggregate) {
            const int n_local = (npairs > crank) ? (npairs - crank + G - 1) / G : 0;
            for (int e = tid; e < MP; e += blockDim.x) {
                const int m = e / P, pp = e - m * P;
                float acc = 0.f;
                for (int li = 0; li < n_local; ++li)
                    if (slot_model[li] == m) acc += slot_s[li * P + pp];
                part_s[buf * MP + e] = acc;
            }
            if (G > 1) cluster.sync(); else __syncthreads();
            if (p.world == 1) {
                for (int e = tid; e < MP; e += blockDim.x) {
                    const int m = e / P;
                    if (tot_s[m] > 0.f) {
                        float v = 0.f;
                        for (int rk = 0; rk < G; ++rk) v += *(cluster.map_shared_rank(part_s + buf * MP + e, rk));
                        theta_s[e] = v;
                    }
                }
            }
            __syncthreads();
        }
        if (p.world > 1) {
            // ---- cross-GPU exchange, LL protocol (flag-in-data, like NCCL's LL): every 8-byte inbox word is
            //      {partial value, round epoch} written by ONE st.v2 — no fence, no separate flag, no round trip: the cost is
            //      one one-way NVLink store latency.  CTA k of the cluster serves the destinations g ≡ k (mod G); every CTA
            //      polls this rank's own inbox (local L2) and sums the senders in rank order (bit-identical on all ranks).
            //      Slots are double-buffered by epoch parity: a sender can only reach epoch E+2 after it has received E+1
            //      from every rank, i.e. after every rank finished reading E.  With skip_aggregate the exchange still runs
            //      (zeros) so that ranks stay within one round of each other (the metrics staging below relies on it).
            const unsigned epoch = flag_base + (unsigned)r + 1u;
            const int xbuf = (int)((flag_base + (unsigned)r) & 1u);
            const size_t slot = (size_t)(xbuf * p.world + p.rank) * MP;
            for (int e = tid; e < MP; e += blockDim.x) {
                float v = 0.f;
                if (!p.skip_aggregate)
                    for (int rk = 0; rk < G; ++rk) v += *(cluster.map_shared_rank(part_s + buf * MP + e, rk));
                for (int gq = crank; gq < p.world; gq += G)
                    st_ll(reinterpret_cast<uint2*>(p.inbox[gq]) + slot + e, v, epoch);
            }
            const uint2* inb = reinterpret_cast<const uint2*>(p.inbox[p.rank]) + (size_t)(xbuf * p.world) * MP;
            SpinGuard sg;
            for (int e = tid; e < MP; e += blockDim.x) {
                uint2 w[kMaxPeers];
#pragma unroll
                for (int gq = 0; gq < kMaxPeers; ++gq)   // all senders' words in flight at once (one L2 latency, not W)
                    if (gq < p.world) w[gq] = ld_ll(inb + (size_t)gq * MP + e);
                float v = 0.f;
                bool ok = true;
#pragma unroll
                for (int gq = 0; gq < kMaxPeers; ++gq) {
                    if (gq < p.world) {
                        while (ok && w[gq].y != epoch) {
                            if (sg.expired(p.spin_timeout_ns)) { ok = false; break; }
                            w[gq] = ld_ll(inb + (size_t)gq * MP + e);
                        }
                        v += __uint_as_float(w[gq].x);
                    }
                }
                // a peer that never arrives: raise the (host-visible) error flag and KEEP the old model — never consume a
                // stale or partial inbox; the host raises at its next metrics read (DriftSim._check_peer_error)
                if (!ok) { if (p.error_flag) atomicExch(p.error_flag, 1); }
                else if (!p.skip_aggregate && tot_s[e / P] > 0.f) theta_s[e] = v;
            }
            __syncthreads();
        }
        if (p.timers && crank == 0 && blockIdx.x == 0 && tid == 0) p.timers[r * 4 + 1] = globaltimer_ns();

        // ------------------------------------------------------------------ IFCA: per-round hard re-clustering
        if (p.recluster_hard) {
            for (int c = crank * NW + warp; c < C; c += G * NW) {
                const int ns = p.nsamp[t * C + c];
                int best = 0; float bestc = -1.f;
                for (int m = 0; m < M; ++m) {
                    float th[P];
#pragma unroll
                    for (int q = 0; q < P; ++q) th[q] = theta_s[m * P + q];
                    float corr = 0.f;
                    for (int s = lane; s < ns; s += 32) {
                        const size_t row = (size_t)(t * C + c) * S + s;
                        float x[IN];
#pragma unroll
                        for (int q = 0; q < IN; ++q) x[q] = p.X[row * IN + q];
                        float z[OUT], h[HID > 0 ? HID : 1], pr[OUT];
                        int am;
                        Net::forward(th, x, z, h);
                        Net::softmax_ce(z, p.Y[row], pr, am);
                        corr += (am == p.Y[row]) ? 1.f : 0.f;
                    }
                    corr = warp_sum(corr);
                    if (corr > bestc) { bestc = corr; best = m; }
                }
                if (lane < M || M > 32)
                    for (int m = lane; m < M; m += 32) p.W[(t * M + m) * C + c] = (m == best) ? 1.f : 0.f;
            }
            __threadfence();
            if (G > 1) cluster.sync(); else __syncthreads();
        }

        // ------------------------------------------------------------------ evaluation: one warp per (client, split)
        for (int it = crank * NW + warp; it < 2 * C; it += G * NW) {
            const int c = it >> 1, which = it & 1;
            if (p.world > 1 && (c % p.world) != p.rank) continue;
            const int tt = t + which;
            if (tt >= p.T1) continue;
            int pick = 0; float bw = p.W[(t * M + 0) * C + c];
            for (int m = 1; m < M; ++m) { const float w = p.W[(t * M + m) * C + c]; if (w > bw) { bw = w; pick = m; } }
            int msel = pick;
            const int* ovr = which ? p.eval_test_model : p.eval_train_model;
            if (ovr && ovr[c] >= 0) msel = ovr[c];
            const int ns = p.nsamp[tt * C + c];
            float corr = 0.f, loss = 0.f;
            if (which == 1 && p.ens_mode != 0) {
                for (int sx = lane; sx < ns; sx += 32) {
                    const size_t row = (size_t)(tt * C + c) * S + sx;
                    float x[IN];
#pragma unroll
                    for (int q = 0; q < IN; ++q) x[q] = p.X[row * IN + q];
                    float tally[OUT];
#pragma unroll
                    for (int o = 0; o < OUT; ++o) tally[o] = 0.f;
                    for (int m = 0; m < M; ++m) {
                        const float w = p.ens_w[c * M + m];
                        if (!(w > 0.f)) continue;
                        float th[P];
#pragma unroll
                        for (int q = 0; q < P; ++q) th[q] = theta_s[m * P + q];
                        float z[OUT], h[HID > 0 ? HID : 1], pr[OUT];
                        int am;
                        Net::forward(th, x, z, h);
                        Net::softmax_ce(z, 0, pr, am);
#pragma unroll
                        for (int o = 0; o < OUT; ++o) tally[o] += (p.ens_mode == 1) ? ((o == am) ? w : 0.f) : w * pr[o];
                    }
                    int am = 0; float mx = tally[0];
#pragma unroll
                    for (int o = 1; o < OUT; ++o) if (tally[o] > mx) { mx = tally[o]; am = o; }
                    corr += (am == p.Y[row]) ? 1.f : 0.f;
                }
            } else {
                float th[P];
#pragma unroll
                for (int q = 0; q < P; ++q) th[q] = theta_s[msel * P + q];
                for (int sx = lane; sx < ns; sx += 32) {
                    const size_t row = (size_t)(tt * C + c) * S + sx;
                    float x[IN];
#pragma unroll
                    for (int q = 0; q < IN; ++q) x[q] = p.X[row * IN + q];
                    const int y = p.Y[row];
                    float z[OUT], h[HID > 0 ? HID : 1], pr[OUT];
                    int am;
                    Net::forward(th, x, z, h);
                    loss += Net::softmax_ce(z, y, pr, am);
                    corr += (am == y) ? 1.f : 0.f;
                }
            }
            corr = warp_sum(corr); loss = warp_sum(loss);
            if (lane == 0) {
                const size_t moff = ((size_t)r * C + c) * 4 + which * 2;
                if (p.world > 1 && p.metrics_peer[0]) {
                    // the owner pushes this client's (correct, loss) pair into EVERY rank's LL staging area as one 16-byte
                    // store {corr, epoch, loss, epoch}; the tail of the launch compacts the staging area into p.metrics
                    const unsigned epoch = flag_base + (unsigned)r + 1u;
                    for (int gq = 0; gq < p.world; ++gq)
                        st_ll2(reinterpret_cast<uint4*>(p.metrics_peer[gq]) + (moff >> 1), corr, loss, epoch);
                } else {
                    *reinterpret_cast<float2*>(p.metrics + moff) = make_float2(corr, loss);
                }
                if (p.host_metrics && p.world == 1) {   // fused D2H: posted writes over PCIe, visible to the host when the kernel retires
                    st_relaxed_sys_f32(p.host_metrics + moff, corr);
                    st_relaxed_sys_f32(p.host_metrics + moff + 1, loss);
                }
            }
        }
        if (p.timers && crank == 0 && blockIdx.x == 0 && tid == 0) p.timers[r * 4 + 2] = globaltimer_ns();
        // (no barrier needed here: θ_s is next written after the __syncthreads that follows local training)
    }

    // ---- multi-GPU: gather the launch's metric rows.  Every (round, client, split) pair arrives as one self-validating
    //      16-byte LL word from its owner; cluster rank 0 polls this rank's staging area (one-way NVLink latency after the
    //      slowest peer's evaluation — no fence / flag handshake) and writes the plain [rounds, C, 4] metrics tensor and,
    //      for the end-to-end graph, the pinned host mirror (posted PCIe writes).
    if (p.world > 1 && p.metrics_peer[0] && crank == 0) {
        const uint4* stg = reinterpret_cast<const uint4*>(p.metrics_peer[p.rank]);
        SpinGuard sg;
        for (int e = tid; e < p.rounds * C * 2; e += blockDim.x) {
            const int c = (e >> 1) % C, which = e & 1;
            if (t + which >= p.T1) continue;   // nobody evaluates a test split beyond the last time step
            const unsigned epoch = flag_base + (unsigned)(e / (2 * C)) + 1u;
            (void)c;
            uint4 w = ld_ll2(stg + e);
            bool ok = true;
            while (w.y != epoch || w.w != epoch) {
                if (sg.expired(p.spin_timeout_ns)) { ok = false; break; }
                w = ld_ll2(stg + e);
            }
            if (!ok) { if (p.error_flag) atomicExch(p.error_flag, 2); continue; }
            const float2 v = make_float2(__uint_as_float(w.x), __uint_as_float(w.z));
            *reinterpret_cast<float2*>(p.metrics + 2 * (size_t)e) = v;
            if (p.host_metrics) {
                st_relaxed_sys_f32(p.host_metrics + 2 * (size_t)e, v.x);
                st_relaxed_sys_f32(p.host_metrics + 2 * (size_t)e + 1, v.y);
            }
        }
    }
    if (p.counters && crank == 0 && tid == 0) { p.counters[0] = round0 + p.rounds; p.counters[1] = (int)(flag_base + (unsigned)p.rounds); }
    // ---- write the models back (all CTAs hold identical copies; cluster rank 0 stores) ----
    __syncthreads();
    if (crank == 0)
        for (int e = tid; e < MP; e += blockDim.x) p.theta[(e / P) * p.theta_stride + (e % P)] = theta_s[e];
    if (G > 1) cluster.sync();  // keep every CTA's smem alive until all DSMEM reads are done
}

// ================================================================================ standalone K4: eval matrix
template <class Net>
__global__ void mlp_eval_matrix_kernel(const float* __restrict__ theta, int theta_stride, int M, const float* __restrict__ X,
                                       const int* __restrict__ Y, const int* __restrict__ nsamp, int C, int S,
                                       float* __restrict__ correct, float* __restrict__ loss, float* __restrict__ sqerr) {
    constexpr int P = Net::P, IN = Net::kIn, OUT = Net::kOut, HID = Net::kHid;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (gw >= M * C) return;
    const int m = gw / C, c = gw % C;
    float th[P];
#pragma unroll
    for (int q = 0; q < P; ++q) th[q] = theta[(size_t)m * theta_stride + q];
    const int ns = nsamp[c];
    float corr = 0.f, ls = 0.f, sq = 0.f;
    for (int s = lane; s < ns; s += 32) {
        const size_t row = (size_t)c * S + s;
        float x[IN];
#pragma unroll
        for (int q = 0; q < IN; ++q) x[q] = X[row * IN + q];
        const int y = Y[row];
        float z[OUT], h[HID > 0 ? HID : 1], pr[OUT];
        int am;
        Net::forward(th, x, z, h);
        ls += Net::softmax_ce(z, y, pr, am);
        corr += (am == y) ? 1.f : 0.f;
        float py = 0.f;
#pragma unroll
        for (int o = 0; o < OUT; ++o) py = (o == y) ? pr[o] : py;
        sq += (1.f - py) * (1.f - py);
    }
    corr = warp_sum(corr); ls = warp_sum(ls); sq = warp_sum(sq);
    if (lane == 0) {
        correct[gw] = corr;
        loss[gw] = ls;
        if (sqerr) sqerr[gw] = sq;
    }
}

// ================================================================================ host launchers
// Cluster size and dynamic shared memory of a launch over `slots` worker slots (C, or K with a participants table).  The
// per-CTA staging of trained pairs holds ceil(slots·M / G) rows, so a small requested cluster can overflow 227 KB where a
// larger one fits: the cluster grows (portable sizes, up to 8) until the layout fits.  smem > 227 KB means it never does.
template <class Net>
static int launch_shape(int C, int M, int slots, int cluster, int warps_per_pair, int* smem_out) {
    using Cfg = SmallCfg<Net>;
    const int rows = slots * M;
    const int wpp = (warps_per_pair == 4 || warps_per_pair == 2) ? warps_per_pair : 1;
    const int groups_per_cta = Cfg::kWarps / wpp;
    int G = cluster;
    if (G <= 0) {  // auto: enough warp groups for every candidate pair, portable cluster sizes only
        G = 1;
        while (G < 8 && G * groups_per_cta < rows) G *= 2;
    }
    if (G > 8) G = 8;
    auto footprint = [&](int g) { return make_layout<Net>(M, C, (rows + g - 1) / g).total * (int)sizeof(float); };
    int smem = footprint(G);
    while (smem > 227 * 1024 && G < 8) {
        G = (2 * G < 8) ? 2 * G : 8;
        smem = footprint(G);
    }
    *smem_out = smem;
    return G;
}

template <class Net>
static int launch_round(const RoundParams& p, int cluster, cudaStream_t stream, SmallLaunchInfo* info) {
    using Cfg = SmallCfg<Net>;
    int smem = 0;
    const int G = launch_shape<Net>(p.C, p.M, p.participants ? p.K : p.C, cluster, p.warps_per_pair, &smem);
    if (smem > 227 * 1024) return -2;
    auto kern = p.participants ? fed_round_small_kernel<Net, true> : fed_round_small_kernel<Net, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return -3;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(G);
    cfg.blockDim = dim3(Cfg::kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = G;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, kern, p);
    if (info) { info->threads = Cfg::kThreads; info->cluster = G; info->smem_bytes = smem; }
    return e == cudaSuccess ? 0 : -4;
}

int fed_round_small_launch(int kind, int din, int hid, int dout, const RoundParams& p, int cluster, cudaStream_t stream,
                           SmallLaunchInfo* info) {
#define FDB_CASE(K, I, H, O) \
    if (kind == K && din == I && (K == 0 || hid == H) && dout == O) return launch_round<Mlp<K, I, H, O>>(p, cluster, stream, info);
    FDB_MLP_SHAPES(FDB_CASE)
#undef FDB_CASE
    return -1;
}

int fed_round_small_launch_shape(int kind, int din, int hid, int dout, int C, int M, int slots, int cluster,
                                 int warps_per_pair, int* smem) {
#define FDB_CASE(K, I, H, O) \
    if (kind == K && din == I && (K == 0 || hid == H) && dout == O) return launch_shape<Mlp<K, I, H, O>>(C, M, slots, cluster, warps_per_pair, smem);
    FDB_MLP_SHAPES(FDB_CASE)
#undef FDB_CASE
    return -1;
}

template <class Net>
static int fits_round(int C, int M) {
    const int CM = C * M, G = 8;   // the launcher may use up to the portable cluster size
    const SmemLayout L = make_layout<Net>(M, C, (CM + G - 1) / G);
    return L.total * (int)sizeof(float) <= 227 * 1024;
}

// 1 when the fused kernel can run this federation: instantiated shape, t_cur < kTmax, shared-memory layout within 227 KB
int fed_round_small_fits(int kind, int din, int hid, int dout, int C, int M, int t_cur) {
    if (t_cur >= kTmax) return 0;
#define FDB_CASE(K, I, H, O) \
    if (kind == K && din == I && (K == 0 || hid == H) && dout == O) return fits_round<Mlp<K, I, H, O>>(C, M);
    FDB_MLP_SHAPES(FDB_CASE)
#undef FDB_CASE
    return 0;
}

int fed_round_small_supported(int kind, int din, int hid, int dout) {
#define FDB_CASE(K, I, H, O) \
    if (kind == K && din == I && (K == 0 || hid == H) && dout == O) return 1;
    FDB_MLP_SHAPES(FDB_CASE)
#undef FDB_CASE
    return 0;
}

int mlp_eval_matrix_launch(int kind, int din, int hid, int dout, const float* theta, int theta_stride, int M, const float* X,
                           const int* Y, const int* nsamp, int C, int S, float* correct, float* loss, float* sqerr,
                           cudaStream_t stream) {
    const int warps = M * C, threads = 128;
    const int blocks = (warps * 32 + threads - 1) / threads;
#define FDB_CASE(K, I, H, O)                                                                                          \
    if (kind == K && din == I && (K == 0 || hid == H) && dout == O) {                                                  \
        mlp_eval_matrix_kernel<Mlp<K, I, H, O>><<<blocks, threads, 0, stream>>>(theta, theta_stride, M, X, Y, nsamp, C, S, \
                                                                                correct, loss, sqerr);                  \
        return cudaGetLastError() == cudaSuccess ? 0 : -4;                                                            \
    }
    FDB_MLP_SHAPES(FDB_CASE)
#undef FDB_CASE
    return -1;
}

}  // namespace fdb
