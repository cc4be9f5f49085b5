// phendiff_b200 — the training step behind the C ABI (SURVEY §8 row f2): forward + backward of the conditional UNet for one batch
// and the loss of the reference's `_diffusion_and_backward` (src/utils_training.py:374-456), gradient clipping, AdamW and EMA
// (train.py:279-285, utils_training.py:224-241, :439).
//
// fp32 path (this file + pd_train_kernels.cu): NHWC fp32 activations, every forward tensor kept (bump allocation, no reuse), a
// tape of backward closures played in reverse — the graph walk mirrors CustomCondUNet2DModel.forward (cond_unet_2d.py:244-362)
// exactly as the inference recorder in pd_api.cu does.  Parameters and gradients are FLAT fp32 vectors in parameter-table
// order (diffusers checkpoint naming, PyTorch layouts: OIHW convolutions, (out, in) linears), owned by the caller: the Python
// side views them as the module's parameters / .grad, hands the gradient vector to NCCL as one buffer, and the optimiser kernel
// updates the vector in place.  Gradients are ACCUMULATED (+=): the caller zeroes them (optimizer.zero_grad()).
#include "pd_model.h"
#include "pd_train.h"

namespace pd {

struct TT {   // an NHWC fp32 activation and its gradient
    float* d = nullptr;
    float* g = nullptr;
    int C = 0, H = 0, W = 0;
    double* stats = nullptr;   // GroupNorm chunk statistics (computed on first use)
    void* h = nullptr;         // 16-bit copy feeding the tensor-core convolutions (mixed-precision mode; made on first use)
    bool only16 = false;
    void* g16 = nullptr;       // 16-bit-only tensors (GroupNorm outputs whose single consumer is a tensor-core conv: d == g == null): the
                               // gradient the consumer's dgrad writes directly
};

}  // namespace pd

using namespace pd;

struct pd_train {
    pd_unet* m = nullptr;
    int B = 0, H = 0, W = 0;
    std::map<const Param*, size_t> poff;
    std::vector<size_t> poff_by_index;
    size_t nflat = 0;
    size_t act_bytes = 0, aux_bytes = 0, ws_bytes = 0;
    uint8_t* ws = nullptr;
    // per step
    bool dry = true;
    size_t act_bump = 0, aux_bump = 0;
    std::vector<std::function<int(cudaStream_t)>> tape;
    std::vector<std::unique_ptr<TT>> tts;
    const float* P = nullptr;
    float* G = nullptr;
    cudaStream_t s = nullptr;
    int rc = 0;
    int64_t launches = 0;
    // mixed precision (pd_train_set_precision): 16-bit operands (bf16 or fp16) for the convolutions on the tcgen05 kernels and for
    // attention on mma.sync, everything else fp32
    int dt = DT_F32;
    const float* loss_scale = nullptr;   // device scalar multiplying the loss gradient (pd_train_set_loss_scale); null: 1
    unsigned tc_mask = 127;        // 1 conv forward, 2 dgrad, 4 wgrad, 8 attention, 16 16-bit-only GroupNorm outputs + fused q/k/v, 32 padded
                                   // tensor-core GEMMs for conv_in / conv_out gradients, 64 GroupNorm statistics from the conv's forward
                                   // epilogue (PHENDIFF_B200_TRAIN_TC)
    size_t scr_max = 0, wstage_max = 0;          // shared scratch: two 16-bit activation-sized buffers + the wgrad staging tile
    struct ConvSlot { ConvTcDesc d; ConvTcPlan* pl = nullptr; };
    struct WgSlot { WgradTcDesc d; WgradTcPlan* pl = nullptr; };
    std::vector<ConvSlot> conv_plans;
    std::vector<WgSlot> wg_plans;
    size_t conv_cursor = 0, wg_cursor = 0;
    int tc_convs = 0, tc_wgrads = 0;
    // input-gradient-only backward (f4, pd_train_forward / pd_train_backward_input): parameter gradients are skipped (G == null)
    bool param_grads() const { return G != nullptr; }
    float* d_input = nullptr;      // (B, Cin, H, W) fp32 NCHW, written by conv_in's backward when set
    float *pending_mo = nullptr, *pending_dm = nullptr;
    bool forward_pending = false;
    void* scr_a() const { return ws + 2 * act_bytes + aux_bytes - 2 * scr_max - wstage_max; }
    void* scr_b() const { return ws + 2 * act_bytes + aux_bytes - scr_max - wstage_max; }
    float* wstage() const { return (float*)(ws + 2 * act_bytes + aux_bytes - wstage_max); }
    ConvTcPlan* conv_plan(size_t idx, const ConvTcDesc& d, int* rc_out) {
        if (idx >= conv_plans.size()) conv_plans.resize(idx + 1);
        ConvSlot& sl = conv_plans[idx];
        if (sl.pl && memcmp(&sl.d, &d, sizeof(d)) == 0) return sl.pl;
        if (sl.pl) { conv_tc_plan_destroy(sl.pl); sl.pl = nullptr; }
        int r = conv_tc_plan_create(d, &sl.pl);
        if (r) { *rc_out = r; return nullptr; }
        sl.d = d;
        return sl.pl;
    }
    WgradTcPlan* wg_plan(size_t idx, const WgradTcDesc& d, int* rc_out) {
        if (idx >= wg_plans.size()) wg_plans.resize(idx + 1);
        WgSlot& sl = wg_plans[idx];
        if (sl.pl && memcmp(&sl.d, &d, sizeof(d)) == 0) return sl.pl;
        if (sl.pl) { wgrad_tc_plan_destroy(sl.pl); sl.pl = nullptr; }
        int r = wgrad_tc_plan_create(d, &sl.pl);
        if (r) { *rc_out = r; return nullptr; }
        sl.d = d;
        return sl.pl;
    }
    ~pd_train() {
        for (auto& c : conv_plans) if (c.pl) conv_tc_plan_destroy(c.pl);
        for (auto& w : wg_plans) if (w.pl) wgrad_tc_plan_destroy(w.pl);
    }
};

namespace pd {

struct Walk {
    pd_train* t;
    pd_unet* m;
    int B;

    const float* p(const Param* q) const { return t->P ? t->P + t->poff.at(q) : nullptr; }
    float* gr(const Param* q) const { return t->G ? t->G + t->poff.at(q) : nullptr; }
    bool dry() const { return t->dry; }
    cudaStream_t s() const { return t->s; }
    void run(int rc) { if (rc && !t->rc) t->rc = rc; }
    void cu(cudaError_t e) { if (e != cudaSuccess && !t->rc) { set_error(std::string("training step: ") + cudaGetErrorString(e)); t->rc = 2; } }
    void count(int n = 1) { t->launches += n; }
    template <typename F> void bwd(F f) { if (!dry()) t->tape.push_back(f); }

    // activations: data in [0, act_bytes), gradients mirrored at + act_bytes; aux buffers (no gradient mirror) behind both
    TT* act(int C, int H, int W) {
        auto tt = std::make_unique<TT>();
        tt->C = C; tt->H = H; tt->W = W;
        const size_t bytes = (((size_t)B * H * W * C * sizeof(float)) + 255) & ~(size_t)255;
        if (!dry()) {
            tt->d = (float*)(t->ws + t->act_bump);
            tt->g = (float*)(t->ws + t->act_bytes + t->act_bump);
            // every backward operator accumulates into fp32 gradients: they start at zero (16-bit-only tensors are written, not
            // accumulated, and are not cleared)
            cu(cudaMemsetAsync(tt->g, 0, bytes, s()));
        }
        t->act_bump += bytes;
        TT* r = tt.get();
        t->tts.push_back(std::move(tt));
        return r;
    }
    // 16-bit-only activation: data and gradient in the same two regions, half the bytes
    TT* act16(int C, int H, int W) {
        auto tt = std::make_unique<TT>();
        tt->C = C; tt->H = H; tt->W = W; tt->only16 = true;
        const size_t bytes = (((size_t)B * H * W * C * 2) + 255) & ~(size_t)255;
        if (!dry()) {
            tt->h = (void*)(t->ws + t->act_bump);
            tt->g16 = (void*)(t->ws + t->act_bytes + t->act_bump);
        } else {
            tt->h = reinterpret_cast<void*>(uintptr_t(8));
        }
        t->act_bump += bytes;
        TT* r = tt.get();
        t->tts.push_back(std::move(tt));
        return r;
    }
    void* aux(size_t bytes, bool zero = false) {
        bytes = (bytes + 255) & ~(size_t)255;
        void* r = dry() ? nullptr : (void*)(t->ws + 2 * t->act_bytes + t->aux_bump);
        t->aux_bump += bytes;
        if (r && zero) cu(cudaMemsetAsync(r, 0, bytes, s()));
        return r;
    }

    double* stats_of(TT* x) {
        if (!x->stats) {
            x->stats = (double*)aux((size_t)B * (x->C / m->stats_cw) * 2 * sizeof(double), true);
            if (!dry()) {
                run(launch_gn_chunk_stats(DT_F32, x->d, B, x->H * x->W, x->C, m->stats_cw, x->stats, s()));
                count();
            } else {
                x->stats = reinterpret_cast<double*>(uintptr_t(8));   // dry pass: remember that the slot exists
            }
        }
        return x->stats;
    }

    // 16-bit copy of an activation (made once, on first use by a tensor-core convolution)
    void* half_of(TT* x) {
        if (!x->h) {
            const size_t n = (size_t)B * x->H * x->W * x->C;
            x->h = aux(n * 2);
            if (!dry()) { run(launch_f2h(t->dt, x->d, x->h, n, s())); count(); }
            else x->h = reinterpret_cast<void*>(uintptr_t(8));
        }
        return x->h;
    }
    void need_scratch(size_t bytes) { bytes = (bytes + 255) & ~(size_t)255; if (bytes > t->scr_max) t->scr_max = bytes; }

    // which pieces of a stride-1 'same' convolution over ONE source of C channels run on the tensor cores
    struct TcFlags { bool fwd, dgrad, wgrad; bool all() const { return fwd && dgrad && wgrad; } };
    TcFlags tc_flags(int C, int H, int W, int cout, int k) const {
        TcFlags f{false, false, false};
        if (t->dt == DT_F32) return f;
        ConvTcDesc d{};
        d.dt = t->dt; d.C = C; d.N = B; d.H = H; d.W = W; d.ksize = k; d.stride = 1; d.pad = k / 2; d.Ho = H; d.Wo = W; d.Cout = cout;
        d.mode = TC_MODE_STD; d.stats_cw = m->stats_cw;
        f.fwd = (t->tc_mask & 1) && conv_halo_supported(d, nullptr);
        ConvTcDesc g = d;
        g.C = cout; g.Cout = C;
        f.dgrad = (t->tc_mask & 2) && conv_halo_supported(g, nullptr);
        WgradTcDesc wd{};
        wd.dt = t->dt; wd.C1 = C; wd.N = B; wd.H = H; wd.W = W; wd.Cout = cout; wd.ksize = k;
        f.wgrad = (t->tc_mask & 4) && wgrad_tc_supported(wd, nullptr);
        return f;
    }

    // y = act(GroupNorm(concat(a, b))).  to16: the output exists in 16 bits only (its single consumer is a tensor-core convolution
    // that reads it as an operand and whose dgrad writes the 16-bit gradient this backward reads)
    TT* gn(const GNL& g, TT* a, TT* b, bool silu, bool to16 = false) {
        const int C = a->C + (b ? b->C : 0), HW = a->H * a->W;
        to16 = to16 && (t->tc_mask & 16) && C % 8 == 0 && a->C % 8 == 0;
        TT* o = to16 ? act16(C, a->H, a->W) : act(C, a->H, a->W);
        double* st1 = stats_of(a);
        double* st2 = b ? stats_of(b) : nullptr;
        float* gsum = (float*)aux((size_t)B * m->cfg.norm_num_groups * 2 * sizeof(float));
        if (dry()) return o;
        GNBwdArgs ba{};
        ba.x1 = a->d; ba.x2 = b ? b->d : nullptr; ba.dx1 = a->g; ba.dx2 = b ? b->g : nullptr; ba.C1 = a->C; ba.C2 = b ? b->C : 0;
        ba.N = B; ba.HW = HW; ba.groups = m->cfg.norm_num_groups; ba.silu = silu; ba.stats_cw = m->stats_cw; ba.eps = m->cfg.norm_eps; ba.scale = 1.f;
        ba.gamma = p(g.g); ba.beta = p(g.b); ba.dgamma = gr(g.g); ba.dbeta = gr(g.b); ba.stats1 = st1; ba.stats2 = st2; ba.gsum = gsum;
        if (to16) {
            run(launch_gn_apply16(t->dt, ba, o->h, s()));
            ba.dy = o->g16; ba.dy_dt = t->dt;
        } else {
            GNArgs ga{};
            ga.x1 = a->d; ga.x2 = b ? b->d : nullptr; ga.C1 = a->C; ga.C2 = b ? b->C : 0; ga.N = B; ga.HW = HW; ga.groups = m->cfg.norm_num_groups;
            ga.eps = m->cfg.norm_eps; ga.gamma = p(g.g); ga.beta = p(g.b); ga.silu = silu; ga.stats_cw = m->stats_cw; ga.stats1 = st1; ga.stats2 = st2;
            ga.out = o->d;
            run(launch_gn_apply(DT_F32, true, ga, s()));
            ba.dy = o->g; ba.dy_dt = DT_F32;
        }
        count();
        pd_train* tr = t;
        bwd([ba, tr](cudaStream_t st) { tr->launches += 2; return launch_gn_bwd(ba, st); });
        return o;
    }

    // out = (conv(concat(a, b)) + bias + addvec[n] + residual) * out_scale; d_addvec (B, Cout) receives the per-image column sums
    TT* conv(const Param* w, const Param* bias, int cout, int k, int stride, int pad, TT* a, TT* b, const float* addvec, float* d_addvec,
             TT* residual, float out_scale, bool want_stats = true) {
        const int Ct = a->C + (b ? b->C : 0);
        const int Ho = stride == 2 ? a->H / 2 : a->H, Wo = stride == 2 ? a->W / 2 : a->W;
        TT* o = act(cout, Ho, Wo);
        const int kk = k * k;
        // which pieces of this layer run on the tensor cores (mixed-precision mode, shapes the tcgen05 kernels take)
        bool tc_fwd = false, tc_dg[2] = {false, false}, tc_wg = false, tc_dg_s2 = false;
        if (t->dt != DT_F32) {
            ConvTcDesc d{};
            d.dt = t->dt; d.C = Ct; d.C2 = b ? b->C : 0; d.N = B; d.H = a->H; d.W = a->W; d.ksize = k; d.stride = stride; d.pad = pad; d.Ho = Ho; d.Wo = Wo;
            d.Cout = cout; d.mode = TC_MODE_STD; d.stats_cw = m->stats_cw;
            tc_fwd = (t->tc_mask & 1) && (conv_halo_supported(d, nullptr) || (!b && conv_tc_supported(d, nullptr)));
            if (stride == 1 && pad == k / 2) {
                const TT* srcs[2] = {a, b};
                for (int q = 0; q < 2; ++q) {
                    if (!srcs[q]) continue;
                    ConvTcDesc g{};
                    g.dt = t->dt; g.C = cout; g.N = B; g.H = Ho; g.W = Wo; g.ksize = k; g.stride = 1; g.pad = pad; g.Ho = Ho; g.Wo = Wo; g.Cout = srcs[q]->C;
                    g.mode = TC_MODE_STD; g.stats_cw = m->stats_cw;
                    tc_dg[q] = (t->tc_mask & 2) && conv_halo_supported(g, nullptr);
                }
                WgradTcDesc wd{};
                wd.dt = t->dt; wd.C1 = a->C; wd.C2 = b ? b->C : 0; wd.N = B; wd.H = a->H; wd.W = a->W; wd.Cout = cout; wd.ksize = k;
                tc_wg = (t->tc_mask & 4) && wgrad_tc_supported(wd, nullptr);
            } else if (stride == 2 && k == 3 && pad == 1 && !b && a->H == 2 * Ho && a->W == 2 * Wo) {
                WgradTcDesc wd{};
                wd.dt = t->dt; wd.C1 = a->C; wd.N = B; wd.H = a->H; wd.W = a->W; wd.Cout = cout; wd.ksize = 3; wd.stride = 2;
                tc_wg = (t->tc_mask & 4) && wgrad_tc_supported(wd, nullptr);
                // stride-2 dgrad = the halo kernel's sub-pixel phase mode on dY (launch_relayout_tc_dgrad_s2)
                ConvTcDesc g{};
                g.dt = t->dt; g.C = cout; g.N = B; g.H = Ho; g.W = Wo; g.ksize = 3; g.stride = 1; g.pad = 1; g.Ho = a->H; g.Wo = a->W; g.Cout = a->C;
                g.upsample = 1; g.mode = TC_MODE_STD; g.stats_cw = m->stats_cw;
                tc_dg_s2 = (t->tc_mask & 2) && conv_halo_supported(g, nullptr);
            }
        }
        if ((a->only16 && !(tc_fwd && tc_dg[0] && tc_wg)) || (b && b->only16)) {
            set_error("internal: 16-bit-only activation feeding a convolution that is not fully on the tensor-core path"); run(1);
        }
        const bool any_dg_simt = stride == 1 && ((!tc_dg[0]) || (b && !tc_dg[1]));
        float* w_fwd = tc_fwd ? nullptr : (float*)aux((size_t)kk * Ct * cout * sizeof(float));
        float* wd1 = (stride == 1 && !tc_dg[0]) ? (float*)aux((size_t)kk * cout * a->C * sizeof(float)) : nullptr;
        float* wd2 = (stride == 1 && b && !tc_dg[1]) ? (float*)aux((size_t)kk * cout * b->C * sizeof(float)) : nullptr;
        (void)any_dg_simt;
        void* w16 = tc_fwd ? aux((size_t)kk * Ct * cout * 2) : nullptr;
        void* wd16[2] = {tc_dg[0] ? aux((size_t)kk * cout * a->C * 2) : (tc_dg_s2 ? aux((size_t)16 * cout * a->C * 2) : nullptr),
                         (b && tc_dg[1]) ? aux((size_t)kk * cout * b->C * 2) : nullptr};
        void* a16 = (tc_fwd || tc_wg) ? half_of(a) : nullptr;
        void* b16 = (b && (tc_fwd || tc_wg)) ? half_of(b) : nullptr;
        if (tc_fwd || tc_dg[0] || tc_dg[1] || tc_wg || tc_dg_s2) {
            need_scratch((size_t)B * Ho * Wo * cout * 2);
            need_scratch((size_t)B * a->H * a->W * std::max(a->C, b ? b->C : 0) * 2);
        }
        if (tc_wg && (size_t)kk * cout * Ct * sizeof(float) > t->wstage_max) t->wstage_max = (((size_t)kk * cout * Ct * sizeof(float)) + 255) & ~(size_t)255;
        const size_t fwd_idx = t->conv_cursor, dg_idx = t->conv_cursor + 1, wg_idx = t->wg_cursor;
        t->conv_cursor += 3; t->wg_cursor += 1;
        // the GroupNorm that consumes this output needs its chunk statistics: produced by the forward epilogue instead of a separate pass
        const bool fuse_stats = tc_fwd && want_stats && (t->tc_mask & 64) && cout % 8 == 0 && cout / 8 <= 256 && (cout / m->cfg.norm_num_groups) % m->stats_cw == 0;
        if (fuse_stats) {
            o->stats = (double*)aux((size_t)B * (cout / m->stats_cw) * 2 * sizeof(double), true);
            if (dry()) o->stats = reinterpret_cast<double*>(uintptr_t(8));
        }
        if (dry()) return o;
        if ((size_t)cout * Ct * kk != w->numel) { set_error("internal: training conv shape mismatch for " + w->name); run(1); return o; }
        if (tc_fwd) {
            run(launch_relayout_tc(t->dt, p(w), cout, Ct, k, w16, kk * Ct, 0, s()));
            ConvTcDesc d{};
            d.dt = t->dt; d.x = a16; d.C = Ct; d.x2 = b ? b16 : nullptr; d.C2 = b ? b->C : 0; d.N = B; d.H = a->H; d.W = a->W; d.ksize = k; d.stride = stride;
            d.pad = pad; d.Ho = Ho; d.Wo = Wo; d.Cout = cout; d.wmat = w16; d.bias = bias ? p(bias) : nullptr; d.out_scale = 1.f; d.out = t->scr_a();
            d.mode = TC_MODE_STD; d.stats_cw = m->stats_cw;
            int prc = 0;
            ConvTcPlan* pl = t->conv_plan(fwd_idx, d, &prc);
            if (!pl) { run(prc); return o; }
            run(conv_tc_launch(pl, s()));
            if (fuse_stats) run(launch_h2f_epilogue_stats(t->dt, t->scr_a(), addvec, residual ? residual->d : nullptr, out_scale, o->d, B, Ho * Wo, cout,
                                                          m->stats_cw, o->stats, s()));
            else run(launch_h2f_epilogue(t->dt, t->scr_a(), addvec, residual ? residual->d : nullptr, out_scale, o->d, B, Ho * Wo, cout, s()));
            count(3);
            t->tc_convs++;
        } else {
            run(launch_relayout_simt(p(w), cout, Ct, k, w_fwd, s()));
            ConvArgs ca{};
            ca.x1 = a->d; ca.x2 = b ? b->d : nullptr; ca.C1 = a->C; ca.C2 = b ? b->C : 0; ca.N = B; ca.H = a->H; ca.W = a->W; ca.Cout = cout;
            ca.ksize = k; ca.stride = stride; ca.pad = pad; ca.Ho = Ho; ca.Wo = Wo; ca.w = w_fwd; ca.bias = bias ? p(bias) : nullptr;
            ca.addvec = addvec; ca.addvec_stride = cout; ca.residual = residual ? residual->d : nullptr; ca.out_scale = out_scale; ca.out = o->d;
            run(launch_conv_simt(DT_F32, ca, s()));
            count(2);
        }
        const float* pw = p(w);
        float* gw = gr(w);
        float* gb = bias ? gr(bias) : nullptr;
        const int Bn = B;
        pd_train* tr = t;
        const TT A = *a, Bt = b ? *b : TT(), O = *o, R = residual ? *residual : TT();
        const bool hasB = b != nullptr, hasR = residual != nullptr;
        const bool tc_dg0 = tc_dg[0], tc_dg1 = tc_dg[1], tc_wg_plan = tc_wg;
        void* const wd16_0 = wd16[0];
        void* const wd16_1 = wd16[1];
        bwd([=](cudaStream_t st) {
            int rc = 0;
            const size_t on = (size_t)Bn * O.H * O.W * O.C;
            // everything below is the gradient of the pre-scale sum
            if (out_scale != 1.0f && (rc = launch_add_inplace(O.g, O.g, out_scale - 1.0f, on, st))) return rc;
            const int M = Bn * O.H * O.W;
            const int dt = tr->dt;
            const bool need16 = (tc_wg_plan && gw) || tc_dg0 || tc_dg1 || tc_dg_s2;
            float* dav = tr->param_grads() ? d_addvec : nullptr;     // only feeds parameter gradients (time-embedding MLP)
            const bool do_tc_wg = tc_wg_plan && gw != nullptr;
            if (need16 || (O.C % 4 == 0 && O.H * O.W >= 64 && (gb || dav))) {
                // one pass over dY: bias gradient, per-image sums for the time-embedding projection, and the 16-bit copy
                if ((rc = launch_colsum_cast(dt == DT_F32 ? DT_BF16 : dt, O.g, Bn, O.H * O.W, O.C, gb, dav, need16 ? tr->scr_a() : nullptr, st))) return rc;
            } else {
                if (gb && (rc = launch_colsum(O.g, M, O.C, M, 1.f, gb, st))) return rc;
                if (dav && (rc = launch_colsum(O.g, M, O.C, O.H * O.W, 1.f, dav, st))) return rc;   // per image: (B, Cout)
            }
            if (hasR && R.g && (rc = launch_add_inplace(R.g, O.g, 1.0f, on, st))) return rc;
            if (do_tc_wg) {
                const size_t wbytes = (size_t)kk * O.C * Ct * sizeof(float);
                PD_CHECK_CUDA(cudaMemsetAsync(tr->wstage(), 0, wbytes, st));
                WgradTcDesc wd{};
                wd.dt = dt; wd.x1 = A.h; wd.x2 = hasB ? Bt.h : nullptr; wd.C1 = A.C; wd.C2 = hasB ? Bt.C : 0; wd.N = Bn; wd.H = A.H; wd.W = A.W;
                wd.Cout = O.C; wd.ksize = k; wd.dy = tr->scr_a(); wd.stage = tr->wstage(); wd.stride = stride;
                WgradTcPlan* wp = tr->wg_plan(wg_idx, wd, &rc);
                if (!wp) return rc;
                if ((rc = wgrad_tc_launch(wp, st))) return rc;
                if ((rc = launch_wgrad_unstage(tr->wstage(), O.C, Ct, kk, gw, st))) return rc;
                tr->launches += 3;
                tr->tc_wgrads++;
            } else if (gw) {
                WgradArgs wa{};
                wa.x1 = A.d; wa.x2 = hasB ? Bt.d : nullptr; wa.C1 = A.C; wa.C2 = hasB ? Bt.C : 0; wa.N = Bn; wa.H = A.H; wa.W = A.W; wa.Cout = O.C;
                wa.ksize = k; wa.stride = stride; wa.pad = pad; wa.Ho = O.H; wa.Wo = O.W; wa.dy = O.g; wa.dw = gw; wa.scale = 1.f;
                if ((rc = launch_conv_wgrad(wa, st))) return rc;
                tr->launches += 1;
            }
            tr->launches += 3;
            if (stride == 1) {
                const TT* srcs[2] = {&A, hasB ? &Bt : nullptr};
                float* wds[2] = {wd1, wd2};
                const bool tcd[2] = {tc_dg0, tc_dg1};
                void* const wd16s[2] = {wd16_0, wd16_1};
                int i0 = 0;
                for (int q = 0; q < 2; ++q) {
                    if (!srcs[q]) continue;
                    if (srcs[q]->g16 && tcd[q]) {
                        // 16-bit-only source (a GroupNorm output): the dgrad result IS its gradient, no fp32 accumulation pass
                        if ((rc = launch_relayout_tc_dgrad(dt, pw, O.C, Ct, k, i0, srcs[q]->C, wd16s[q], st))) return rc;
                        ConvTcDesc g{};
                        g.dt = dt; g.x = tr->scr_a(); g.C = O.C; g.N = Bn; g.H = O.H; g.W = O.W; g.ksize = k; g.stride = 1; g.pad = pad; g.Ho = O.H; g.Wo = O.W;
                        g.Cout = srcs[q]->C; g.wmat = wd16s[q]; g.out_scale = 1.f; g.out = srcs[q]->g16; g.mode = TC_MODE_STD; g.stats_cw = tr->m->stats_cw;
                        ConvTcPlan* gp = tr->conv_plan(dg_idx + q, g, &rc);
                        if (!gp) return rc;
                        if ((rc = conv_tc_launch(gp, st))) return rc;
                        tr->launches += 2;
                    } else if (srcs[q]->g && tcd[q]) {
                        // dX = conv(dY, W^T flipped) on the halo kernel, 16-bit result accumulated into the fp32 gradient
                        if ((rc = launch_relayout_tc_dgrad(dt, pw, O.C, Ct, k, i0, srcs[q]->C, wd16s[q], st))) return rc;
                        ConvTcDesc g{};
                        g.dt = dt; g.x = tr->scr_a(); g.C = O.C; g.N = Bn; g.H = O.H; g.W = O.W; g.ksize = k; g.stride = 1; g.pad = pad; g.Ho = O.H; g.Wo = O.W;
                        g.Cout = srcs[q]->C; g.wmat = wd16s[q]; g.out_scale = 1.f; g.out = tr->scr_b(); g.mode = TC_MODE_STD; g.stats_cw = tr->m->stats_cw;
                        ConvTcPlan* gp = tr->conv_plan(dg_idx + q, g, &rc);
                        if (!gp) return rc;
                        if ((rc = conv_tc_launch(gp, st))) return rc;
                        if ((rc = launch_h2f_accumulate(dt, tr->scr_b(), srcs[q]->g, (size_t)Bn * O.H * O.W * srcs[q]->C, st))) return rc;
                        tr->launches += 3;
                    } else if (srcs[q]->g) {
                        if ((rc = launch_relayout_dgrad(pw, O.C, A.C + (hasB ? Bt.C : 0), k, i0, srcs[q]->C, wds[q], st))) return rc;
                        ConvArgs da{};
                        da.x1 = O.g; da.C1 = O.C; da.N = Bn; da.H = O.H; da.W = O.W; da.Cout = srcs[q]->C; da.ksize = k; da.stride = 1;
                        da.pad = k - 1 - pad; da.Ho = O.H; da.Wo = O.W; da.w = wds[q]; da.residual = srcs[q]->g; da.out_scale = 1.f; da.out = srcs[q]->g;
                        if ((rc = launch_conv_simt(DT_F32, da, st))) return rc;
                        tr->launches += 2;
                    }
                    i0 += srcs[q]->C;
                }
            } else if (A.g && tc_dg_s2) {
                if ((rc = launch_relayout_tc_dgrad_s2(dt, pw, O.C, A.C, wd16_0, st))) return rc;
                ConvTcDesc g{};
                g.dt = dt; g.x = tr->scr_a(); g.C = O.C; g.N = Bn; g.H = O.H; g.W = O.W; g.ksize = 3; g.stride = 1; g.pad = 1; g.Ho = A.H; g.Wo = A.W;
                g.Cout = A.C; g.upsample = 1; g.wmat = wd16_0; g.out_scale = 1.f; g.out = tr->scr_b(); g.mode = TC_MODE_STD; g.stats_cw = tr->m->stats_cw;
                ConvTcPlan* gp = tr->conv_plan(dg_idx, g, &rc);
                if (!gp) return rc;
                if ((rc = conv_tc_launch(gp, st))) return rc;
                if ((rc = launch_h2f_accumulate(dt, tr->scr_b(), A.g, (size_t)Bn * A.H * A.W * A.C, st))) return rc;
                tr->launches += 3;
            } else if (A.g) {
                if ((rc = launch_conv_dgrad_gather(O.g, O.C, pw, Bn, A.H, A.W, A.C, O.H, O.W, O.C, pad, stride, A.g, st))) return rc;
                tr->launches += 1;
            }
            return 0;
        });
        return o;
    }

    // ---- time + class embedding (cond_unet_2d.py:289-309) and the per-resnet projections ----
    struct Emb { float *act = nullptr, *dact = nullptr; };
    Emb embedding(const float* timesteps, const int64_t* labels) {
        const int C0 = m->cfg.block_out_channels[0], D = m->D;
        float* e0 = (float*)aux((size_t)B * C0 * sizeof(float));
        float* pre1 = (float*)aux((size_t)B * D * sizeof(float));
        float* h1 = (float*)aux((size_t)B * D * sizeof(float));
        float* emb = (float*)aux((size_t)B * D * sizeof(float));
        Emb e;
        e.act = (float*)aux((size_t)B * D * sizeof(float));
        e.dact = (float*)aux((size_t)B * D * sizeof(float), true);
        float* demb = (float*)aux((size_t)B * D * sizeof(float));
        float* dh1 = (float*)aux((size_t)B * D * sizeof(float));
        float* dpre1 = (float*)aux((size_t)B * D * sizeof(float));
        if (dry()) return e;
        const float *w1 = p(m->te_w1), *b1 = p(m->te_b1), *w2 = p(m->te_w2), *b2 = p(m->te_b2);
        const float* table = (m->cls && labels) ? p(m->cls) : nullptr;
        run(launch_sinusoid(timesteps, B, C0, m->cfg.flip_sin_to_cos, m->cfg.freq_shift, e0, s()));
        run(launch_sgemm(0, 1, B, D, C0, 1.f, e0, C0, w1, C0, pre1, D, 0, s()));
        run(launch_bias_silu_fwd(pre1, b1, nullptr, nullptr, B, D, h1, s()));
        run(launch_sgemm(0, 1, B, D, D, 1.f, h1, D, w2, D, emb, D, 0, s()));
        run(launch_bias_silu_fwd(emb, b2, table, labels, B, D, e.act, s()));
        count(5);
        float *gw1 = gr(m->te_w1), *gb1 = gr(m->te_b1), *gw2 = gr(m->te_w2), *gb2 = gr(m->te_b2);
        float* gcls = table ? gr(m->cls) : nullptr;
        const int Bn = B;
        float* dact = e.dact;
        pd_train* tr = t;
        bwd([=](cudaStream_t st) {
            int rc = 0;
            if (!tr->param_grads()) return 0;     // the embedding branch only reaches parameters (timesteps / labels carry no gradient)
            if ((rc = launch_silu_bwd(emb, dact, (size_t)Bn * D, demb, st))) return rc;
            if (gcls && (rc = launch_scatter_rows(demb, labels, Bn, D, 1.f, gcls, st))) return rc;
            if ((rc = launch_colsum(demb, Bn, D, Bn, 1.f, gb2, st))) return rc;
            if ((rc = launch_sgemm(1, 0, D, D, Bn, 1.f, demb, D, h1, D, gw2, D, 1, st))) return rc;       // dW2 += demb^T h1
            if ((rc = launch_sgemm(0, 0, Bn, D, D, 1.f, demb, D, w2, D, dh1, D, 0, st))) return rc;        // dh1 = demb W2
            if ((rc = launch_silu_bwd(pre1, dh1, (size_t)Bn * D, dpre1, st))) return rc;
            if ((rc = launch_colsum(dpre1, Bn, D, Bn, 1.f, gb1, st))) return rc;
            if ((rc = launch_sgemm(1, 0, D, C0, Bn, 1.f, dpre1, D, e0, C0, gw1, C0, 1, st))) return rc;   // dW1 += dpre1^T e0
            tr->launches += 8;
            return 0;
        });
        return e;
    }
    // temb_r (B, cout) = act W_r^T + b_r; returns the table and its gradient table (filled by the conv that adds it)
    void temb_proj(const ResL& R, const Emb& e, float** temb, float** dtemb) {
        const int D = m->D, co = R.cout;
        *temb = (float*)aux((size_t)B * co * sizeof(float));
        *dtemb = (float*)aux((size_t)B * co * sizeof(float), true);
        if (dry()) return;
        const float *tw = p(R.tw), *tb = p(R.tb);
        run(launch_sgemm(0, 1, B, co, D, 1.f, e.act, D, tw, D, *temb, co, 0, s()));
        run(launch_add_bias_rows(*temb, tb, B, co, s()));
        count(2);
        float *gtw = gr(R.tw), *gtb = gr(R.tb), *dt = *dtemb, *dact = e.dact;
        const float* actp = e.act;
        const int Bn = B;
        pd_train* tr = t;
        bwd([=](cudaStream_t st) {
            int rc = 0;
            if (!tr->param_grads()) return 0;
            if ((rc = launch_colsum(dt, Bn, co, Bn, 1.f, gtb, st))) return rc;
            if ((rc = launch_sgemm(1, 0, co, D, Bn, 1.f, dt, co, actp, D, gtw, D, 1, st))) return rc;     // dW_r += dtemb^T act
            if ((rc = launch_sgemm(0, 0, Bn, D, co, 1.f, dt, co, tw, D, dact, D, 1, st))) return rc;      // dact += dtemb W_r
            tr->launches += 3;
            return 0;
        });
    }

    // ResnetBlock2D (SURVEY A.1) on concat(a, b)
    TT* resnet(const ResL& R, TT* a, TT* b, float* temb, float* dtemb) {
        const int Cin = a->C + (b ? b->C : 0);
        TT* hn = gn(R.n1, a, b, true, tc_flags(Cin, a->H, a->W, R.cout, 3).all());
        TT* h1 = conv(R.c1.w, R.c1.b, R.cout, 3, 1, 1, hn, nullptr, temb, dtemb, nullptr, 1.f);
        TT* h1n = gn(R.n2, h1, nullptr, true, tc_flags(R.cout, a->H, a->W, R.cout, 3).all());
        TT* res = a;
        if (R.has_sc) res = conv(R.sc.w, R.sc.b, R.cout, 1, 1, 0, a, b, nullptr, nullptr, nullptr, 1.f);
        return conv(R.c2.w, R.c2.b, R.cout, 3, 1, 1, h1n, nullptr, nullptr, nullptr, res, 1.0f / R.scale);
    }

    // q, k, v projections as ONE C -> 3C GEMM on the tensor cores (three parameter tensors, one operand): the GroupNorm output has a single
    // consumer, so it can live in 16 bits only and its gradient is the one dgrad's output
    TT* qkv_fused(const AttnL& A, TT* xn) {
        const int C = A.C, H = xn->H, W = xn->W, HW = H * W, C3 = 3 * C;
        TT* o = act(C3, H, W);
        void* w16 = aux((size_t)C3 * C * 2);
        void* wd16 = aux((size_t)C * C3 * 2);
        float* bias3 = (float*)aux((size_t)C3 * sizeof(float));
        float* btmp = (float*)aux((size_t)C3 * sizeof(float));
        void* x16 = half_of(xn);
        need_scratch((size_t)B * HW * C3 * 2);
        if ((size_t)C3 * C * sizeof(float) > t->wstage_max) t->wstage_max = (((size_t)C3 * C * sizeof(float)) + 255) & ~(size_t)255;
        const size_t fwd_idx = t->conv_cursor, dg_idx = t->conv_cursor + 1, wg_idx = t->wg_cursor;
        t->conv_cursor += 2; t->wg_cursor += 1;
        if (dry()) return o;
        const Param* ws[3] = {A.qw, A.kw, A.vw};
        const Param* bs[3] = {A.qb, A.kb, A.vb};
        const int dt = t->dt;
        for (int j = 0; j < 3; ++j) {
            run(launch_relayout_tc(dt, p(ws[j]), C, C, 1, (uint8_t*)w16 + (size_t)j * C * C * 2, C, 0, s()));
            cu(cudaMemcpyAsync(bias3 + j * C, p(bs[j]), C * sizeof(float), cudaMemcpyDeviceToDevice, s()));
        }
        ConvTcDesc d{};
        d.dt = dt; d.x = x16; d.C = C; d.N = B; d.H = H; d.W = W; d.ksize = 1; d.stride = 1; d.pad = 0; d.Ho = H; d.Wo = W; d.Cout = C3; d.wmat = w16;
        d.bias = bias3; d.out_scale = 1.f; d.out = t->scr_a(); d.mode = TC_MODE_STD; d.stats_cw = m->stats_cw;
        int prc = 0;
        ConvTcPlan* pl = t->conv_plan(fwd_idx, d, &prc);
        if (!pl) { run(prc); return o; }
        run(conv_tc_launch(pl, s()));
        run(launch_h2f_epilogue(dt, t->scr_a(), nullptr, nullptr, 1.f, o->d, B, HW, C3, s()));
        count(8);
        t->tc_convs++;
        pd_train* tr = t;
        const TT X = *xn, O = *o;
        const int Bn = B;
        const float* pw[3] = {p(ws[0]), p(ws[1]), p(ws[2])};
        float* gw[3] = {gr(ws[0]), gr(ws[1]), gr(ws[2])};
        float* gb[3] = {gr(bs[0]), gr(bs[1]), gr(bs[2])};
        const float *pw0 = pw[0], *pw1 = pw[1], *pw2 = pw[2];
        float *gw0 = gw[0], *gw1 = gw[1], *gw2 = gw[2], *gb0 = gb[0], *gb1 = gb[1], *gb2 = gb[2];
        bwd([=](cudaStream_t st) {
            int rc = 0;
            const float* pws[3] = {pw0, pw1, pw2};
            float* gws[3] = {gw0, gw1, gw2};
            float* gbs[3] = {gb0, gb1, gb2};
            const bool pg = gw0 != nullptr;
            if (pg) PD_CHECK_CUDA(cudaMemsetAsync(btmp, 0, (size_t)C3 * sizeof(float), st));
            if ((rc = launch_colsum_cast(dt, O.g, Bn, HW, C3, pg ? btmp : nullptr, nullptr, tr->scr_a(), st))) return rc;
            if (pg) {
                for (int j = 0; j < 3; ++j)
                    if ((rc = launch_add_inplace(gbs[j], btmp + j * C, 1.0f, (size_t)C, st))) return rc;
                PD_CHECK_CUDA(cudaMemsetAsync(tr->wstage(), 0, (size_t)C3 * C * sizeof(float), st));
                WgradTcDesc wd{};
                wd.dt = dt; wd.x1 = X.h; wd.C1 = C; wd.N = Bn; wd.H = H; wd.W = W; wd.Cout = C3; wd.ksize = 1; wd.dy = tr->scr_a(); wd.stage = tr->wstage();
                WgradTcPlan* wp = tr->wg_plan(wg_idx, wd, &rc);
                if (!wp) return rc;
                if ((rc = wgrad_tc_launch(wp, st))) return rc;
                for (int j = 0; j < 3; ++j)
                    if ((rc = launch_wgrad_unstage(tr->wstage() + (size_t)j * C * C, C, C, 1, gws[j], st))) return rc;
            }
            for (int j = 0; j < 3; ++j)
                if ((rc = launch_relayout_tc_dgrad(dt, pws[j], C, C, 1, 0, C, wd16, st, C3, j * C))) return rc;
            ConvTcDesc g{};
            g.dt = dt; g.x = tr->scr_a(); g.C = C3; g.N = Bn; g.H = H; g.W = W; g.ksize = 1; g.stride = 1; g.pad = 0; g.Ho = H; g.Wo = W; g.Cout = C;
            g.wmat = wd16; g.out_scale = 1.f; g.out = X.g16 ? X.g16 : tr->scr_b(); g.mode = TC_MODE_STD; g.stats_cw = tr->m->stats_cw;
            ConvTcPlan* gp = tr->conv_plan(dg_idx, g, &rc);
            if (!gp) return rc;
            if ((rc = conv_tc_launch(gp, st))) return rc;
            if (!X.g16 && (rc = launch_h2f_accumulate(dt, tr->scr_b(), X.g, (size_t)Bn * HW * C, st))) return rc;
            tr->launches += 16;
            tr->tc_wgrads++;
            return 0;
        });
        return o;
    }

    // Attention (SURVEY A.2), head_dim 8
    TT* attention(const AttnL& A, TT* x) {
        const int C = A.C, S = x->H * x->W;
        const bool fused = (t->tc_mask & 16) && tc_flags(C, x->H, x->W, 3 * C, 1).all();
        TT* xn = gn(A.gn, x, nullptr, false, fused);
        const float *qd, *kd, *vd;
        float *qg, *kg, *vg;
        int pitch = C;
        if (fused) {
            TT* qkv = qkv_fused(A, xn);
            need_scratch((size_t)B * S * C * 2);
            qd = qkv->d; kd = qkv->d ? qkv->d + C : nullptr; vd = qkv->d ? qkv->d + 2 * C : nullptr;
            qg = qkv->g; kg = qkv->g ? qkv->g + C : nullptr; vg = qkv->g ? qkv->g + 2 * C : nullptr;
            pitch = 3 * C;
        } else {
            TT* q = conv(A.qw, A.qb, C, 1, 1, 0, xn, nullptr, nullptr, nullptr, nullptr, 1.f, false);
            TT* k = conv(A.kw, A.kb, C, 1, 1, 0, xn, nullptr, nullptr, nullptr, nullptr, 1.f, false);
            TT* v = conv(A.vw, A.vb, C, 1, 1, 0, xn, nullptr, nullptr, nullptr, nullptr, 1.f, false);
            qd = q->d; kd = k->d; vd = v->d; qg = q->g; kg = k->g; vg = v->g;
        }
        TT* o = act(C, x->H, x->W);
        float* lse = (float*)aux((size_t)B * (C / 8) * S * sizeof(float));
        float* delta = (float*)aux((size_t)B * (C / 8) * S * sizeof(float));
        if (!dry()) {
            const bool mma = t->dt != DT_F32 && (t->tc_mask & 8) && attn8_mma_supported(S, C, pitch);
            run(mma ? launch_attn8_mma_fwd(t->dt, qd, kd, vd, pitch, B, S, C, o->d, lse, s()) : launch_attn8_fwd(qd, kd, vd, pitch, B, S, C, o->d, lse, s()));
            count();
            const TT O = *o;
            const int Bn = B;
            pd_train* tr = t;
            bwd([=](cudaStream_t st) {
                tr->launches += 2;
                return mma ? launch_attn8_mma_bwd(tr->dt, qd, kd, vd, pitch, O.d, O.g, lse, Bn, S, C, qg, kg, vg, delta, st)
                           : launch_attn8_bwd(qd, kd, vd, pitch, O.d, O.g, lse, Bn, S, C, qg, kg, vg, delta, st);
            });
        }
        return conv(A.ow, A.ob, C, 1, 1, 0, o, nullptr, nullptr, nullptr, x, 1.0f / A.rescale);
    }

    TT* upsample(TT* x) {
        TT* o = act(x->C, 2 * x->H, 2 * x->W);
        if (dry()) return o;
        run(launch_upsample2x(DT_F32, x->d, B, x->H, x->W, x->C, o->d, s()));
        count();
        const TT X = *x, O = *o;
        const int Bn = B;
        pd_train* tr = t;
        bwd([=](cudaStream_t st) { tr->launches += 1; return launch_upsample2x_bwd(O.g, Bn, X.H, X.W, X.C, X.g, st); });
        return o;
    }

    // whole forward; returns the NCHW fp32 model output (aux) and registers every backward closure
    float* forward(const float* noisy, const float* timesteps, const int64_t* labels, float** dm_out) {
        const pd_unet_config_t& c = m->cfg;
        const int H = t->H, W = t->W, C0 = c.block_out_channels[0], Cin = c.in_channels, Cout = c.out_channels;
        Emb e = embedding(timesteps, labels);
        std::vector<std::pair<float*, float*>> tembs;   // per resnet in graph order
        auto all_res = [&](auto&& f) {
            for (auto& d : m->down) for (auto& r : d.res) f(r);
            f(m->mid_r0); f(m->mid_r1);
            for (auto& u : m->up) for (auto& r : u.res) f(r);
        };
        std::map<const ResL*, std::pair<float*, float*>> temb_of;
        all_res([&](const ResL& r) { float *a = nullptr, *b = nullptr; temb_proj(r, e, &a, &b); temb_of[&r] = {a, b}; });
        // conv_in (cond_unet_2d.py:313): NCHW fp32 -> NHWC
        TT* x = act(C0, H, W);
        float* w_in = (float*)aux((size_t)9 * Cin * C0 * sizeof(float));
        float* xin = (float*)aux((size_t)B * H * W * 4 * sizeof(float));
        // gradients of conv_in / conv_out on the tensor cores: the 3-channel side zero-padded to 128 channels (the wasted MACs are
        // cheaper than the CUDA-core kernels by an order of magnitude)
        constexpr int CP = 128;
        bool tc_in = false, tc_out = false;
        if (t->dt != DT_F32 && (t->tc_mask & 32) && Cin <= CP && Cout <= CP) {
            WgradTcDesc wi{};
            wi.dt = t->dt; wi.C1 = CP; wi.N = B; wi.H = H; wi.W = W; wi.Cout = C0; wi.ksize = 3;
            tc_in = wgrad_tc_supported(wi, nullptr);
            WgradTcDesc wo{};
            wo.dt = t->dt; wo.C1 = C0; wo.N = B; wo.H = H; wo.W = W; wo.Cout = CP; wo.ksize = 3;
            ConvTcDesc g{};
            g.dt = t->dt; g.C = CP; g.N = B; g.H = H; g.W = W; g.ksize = 3; g.stride = 1; g.pad = 1; g.Ho = H; g.Wo = W; g.Cout = C0; g.mode = TC_MODE_STD;
            g.stats_cw = m->stats_cw;
            tc_out = wgrad_tc_supported(wo, nullptr) && conv_halo_supported(g, nullptr);
        }
        void* pad16 = (tc_in || tc_out) ? aux((size_t)B * H * W * CP * 2) : nullptr;     // padded operand (conv_out: dY, then conv_in: X)
        void* wd16_out = tc_out ? aux((size_t)C0 * 9 * CP * 2) : nullptr;
        if (tc_in || tc_out) {
            need_scratch((size_t)B * H * W * C0 * 2);
            if ((size_t)9 * CP * C0 * sizeof(float) > t->wstage_max) t->wstage_max = (size_t)9 * CP * C0 * sizeof(float);
        }
        const size_t in_wg_idx = t->wg_cursor, out_wg_idx = t->wg_cursor + 1, out_dg_idx = t->conv_cursor, in_dg_idx = t->conv_cursor + 1;
        t->wg_cursor += 2; t->conv_cursor += 2;
        // input gradient of conv_in (f4: torch.autograd.grad(losses, images), utils_Img2Img.py:741): on the halo kernel with the 3 input
        // channels padded to 64 output columns in mixed-precision mode, by the gather kernel on the fp32 path
        bool tc_in_dg = false;
        if (t->dt != DT_F32 && (t->tc_mask & 2) && Cin <= 64) {
            ConvTcDesc g{};
            g.dt = t->dt; g.C = C0; g.N = B; g.H = H; g.W = W; g.ksize = 3; g.stride = 1; g.pad = 1; g.Ho = H; g.Wo = W; g.Cout = 64; g.mode = TC_MODE_STD;
            g.stats_cw = m->stats_cw;
            tc_in_dg = conv_halo_supported(g, nullptr);
        }
        void* wd16_in = tc_in_dg ? aux((size_t)64 * 9 * C0 * 2) : nullptr;
        void* dxin = aux((size_t)B * H * W * (tc_in_dg ? 64 * 2 : Cin * sizeof(float)));      // NHWC staging of the input gradient
        if (tc_in_dg) need_scratch((size_t)B * H * W * C0 * 2);
        if (!dry()) {
            run(launch_relayout_simt(p(m->conv_in.w), C0, Cin, 3, w_in, s()));
            run(launch_conv_in(DT_F32, noisy, w_in, p(m->conv_in.b), B, Cin, H, W, C0, x->d, s()));
            run(launch_nchw_to_nhwc_pad(noisy, B, Cin, H * W, 4, xin, s()));
            count(3);
            const TT X = *x;
            float *gw = gr(m->conv_in.w), *gb = gr(m->conv_in.b);
            const int Bn = B;
            pd_train* tr = t;
            const float* pw_in = p(m->conv_in.w);
            bwd([=](cudaStream_t st) {
                int rc = 0;
                if (tr->d_input) {
                    const int dt = tr->dt;
                    if (tc_in_dg) {
                        if ((rc = launch_f2h(dt, X.g, tr->scr_a(), (size_t)Bn * H * W * C0, st))) return rc;
                        PD_CHECK_CUDA(cudaMemsetAsync(wd16_in, 0, (size_t)64 * 9 * C0 * 2, st));
                        if ((rc = launch_relayout_tc_dgrad(dt, pw_in, C0, Cin, 3, 0, Cin, wd16_in, st))) return rc;
                        ConvTcDesc g{};
                        g.dt = dt; g.x = tr->scr_a(); g.C = C0; g.N = Bn; g.H = H; g.W = W; g.ksize = 3; g.stride = 1; g.pad = 1; g.Ho = H; g.Wo = W; g.Cout = 64;
                        g.wmat = wd16_in; g.out_scale = 1.f; g.out = dxin; g.mode = TC_MODE_STD; g.stats_cw = tr->m->stats_cw;
                        ConvTcPlan* gp = tr->conv_plan(in_dg_idx, g, &rc);
                        if (!gp) return rc;
                        if ((rc = conv_tc_launch(gp, st))) return rc;
                        if ((rc = launch_nhwc_to_nchw_f32(dt, dxin, Bn, Cin, H * W, 64, tr->d_input, st))) return rc;
                    } else {
                        PD_CHECK_CUDA(cudaMemsetAsync(dxin, 0, (size_t)Bn * H * W * Cin * sizeof(float), st));
                        if ((rc = launch_conv_dgrad_gather(X.g, C0, pw_in, Bn, H, W, Cin, H, W, C0, 1, 1, (float*)dxin, st))) return rc;
                        if ((rc = launch_nhwc_to_nchw_f32(DT_F32, dxin, Bn, Cin, H * W, Cin, tr->d_input, st))) return rc;
                    }
                    tr->launches += 4;
                }
                if (!tr->param_grads()) return 0;
                if (tc_in) {
                    const int dt = tr->dt;
                    if ((rc = launch_colsum_cast(dt, X.g, Bn, H * W, C0, gb, nullptr, tr->scr_a(), st))) return rc;
                    if ((rc = launch_nchw_to_nhwc16_pad(dt, noisy, Bn, Cin, H * W, CP, pad16, st))) return rc;
                    PD_CHECK_CUDA(cudaMemsetAsync(tr->wstage(), 0, (size_t)9 * C0 * CP * sizeof(float), st));
                    WgradTcDesc wd{};
                    wd.dt = dt; wd.x1 = pad16; wd.C1 = CP; wd.N = Bn; wd.H = H; wd.W = W; wd.Cout = C0; wd.ksize = 3; wd.dy = tr->scr_a(); wd.stage = tr->wstage();
                    WgradTcPlan* wp = tr->wg_plan(in_wg_idx, wd, &rc);
                    if (!wp) return rc;
                    if ((rc = wgrad_tc_launch(wp, st))) return rc;
                    tr->launches += 5;
                    tr->tc_wgrads++;
                    return launch_wgrad_unstage(tr->wstage(), C0, Cin, 9, gw, st, C0, CP);
                }
                rc = launch_colsum(X.g, Bn * H * W, C0, Bn * H * W, 1.f, gb, st);
                if (rc) return rc;
                WgradArgs wa{};
                wa.x1 = xin; wa.C1 = 4; wa.N = Bn; wa.H = H; wa.W = W; wa.Cout = C0; wa.ksize = 3; wa.stride = 1; wa.pad = 1; wa.Ho = H; wa.Wo = W;
                wa.dy = X.g; wa.dw = gw; wa.scale = 1.f; wa.Iw = Cin;
                tr->launches += 2;
                return launch_conv_wgrad(wa, st);   // (reached only with parameter gradients on)
            });
        }
        std::vector<TT*> skips{x};
        for (auto& d : m->down) {
            for (size_t j = 0; j < d.res.size(); ++j) {
                auto tp = temb_of[&d.res[j]];
                x = resnet(d.res[j], x, nullptr, tp.first, tp.second);
                if (d.has_attn) x = attention(d.attn[j], x);
                skips.push_back(x);
            }
            if (d.has_down) {
                x = conv(d.down.w, d.down.b, d.down.cout, 3, 2, c.downsample_padding, x, nullptr, nullptr, nullptr, nullptr, 1.f);
                skips.push_back(x);
            }
        }
        { auto tp = temb_of[&m->mid_r0]; x = resnet(m->mid_r0, x, nullptr, tp.first, tp.second); }
        if (m->mid_has_attn) x = attention(m->mid_attn, x);
        { auto tp = temb_of[&m->mid_r1]; x = resnet(m->mid_r1, x, nullptr, tp.first, tp.second); }
        for (auto& u : m->up) {
            for (size_t j = 0; j < u.res.size(); ++j) {
                TT* sk = skips.back(); skips.pop_back();
                auto tp = temb_of[&u.res[j]];
                x = resnet(u.res[j], x, sk, tp.first, tp.second);
                if (u.has_attn) x = attention(u.attn[j], x);
            }
            if (u.has_up) {
                TT* big = upsample(x);
                x = conv(u.up.w, u.up.b, u.up.cout, 3, 1, 1, big, nullptr, nullptr, nullptr, nullptr, 1.f);
            }
        }
        // conv_norm_out + SiLU + conv_out (cond_unet_2d.py:346-348) -> NCHW fp32
        TT* xn = gn(m->norm_out, x, nullptr, true);
        float* w_out = (float*)aux((size_t)9 * C0 * 4 * sizeof(float));
        float* mo = (float*)aux((size_t)B * Cout * H * W * sizeof(float));
        float* dm = (float*)aux((size_t)B * Cout * H * W * sizeof(float));
        float* dy4 = (float*)aux((size_t)B * H * W * 4 * sizeof(float));
        *dm_out = dm;
        if (tc_out) half_of(xn);
        if (!dry()) {
            run(launch_relayout_convout(p(m->conv_out.w), Cout, C0, w_out, s()));
            ConvOutArgs oa{};
            oa.act = xn->d; oa.w = w_out; oa.bias = p(m->conv_out.b); oa.N = B; oa.H = H; oa.W = W; oa.Cin = C0; oa.Cout = Cout; oa.model_out = mo;
            run(launch_conv_out(DT_F32, oa, s()));
            count(2);
            const TT XN = *xn;
            float *gw = gr(m->conv_out.w), *gb = gr(m->conv_out.b);
            const float* pw = p(m->conv_out.w);
            const int Bn = B;
            pd_train* tr = t;
            bwd([=](cudaStream_t st) {
                int rc = launch_nchw_to_nhwc_pad(dm, Bn, Cout, H * W, 4, dy4, st);
                if (rc) return rc;
                if (gb && (rc = launch_colsum(dy4, Bn * H * W, 4, Bn * H * W, 1.f, gb, st, Cout))) return rc;
                if (tc_out) {
                    const int dt = tr->dt;
                    if ((rc = launch_nchw_to_nhwc16_pad(dt, dm, Bn, Cout, H * W, CP, pad16, st))) return rc;
                    if (gw) {
                        PD_CHECK_CUDA(cudaMemsetAsync(tr->wstage(), 0, (size_t)9 * CP * C0 * sizeof(float), st));
                        WgradTcDesc wd{};
                        wd.dt = dt; wd.x1 = XN.h; wd.C1 = C0; wd.N = Bn; wd.H = H; wd.W = W; wd.Cout = CP; wd.ksize = 3; wd.dy = pad16; wd.stage = tr->wstage();
                        WgradTcPlan* wp = tr->wg_plan(out_wg_idx, wd, &rc);
                        if (!wp) return rc;
                        if ((rc = wgrad_tc_launch(wp, st))) return rc;
                        if ((rc = launch_wgrad_unstage(tr->wstage(), Cout, C0, 9, gw, st, CP, C0))) return rc;
                    }
                    PD_CHECK_CUDA(cudaMemsetAsync(wd16_out, 0, (size_t)C0 * 9 * CP * 2, st));
                    if ((rc = launch_relayout_tc_dgrad(dt, pw, Cout, C0, 3, 0, C0, wd16_out, st, 9 * CP, 0, CP))) return rc;
                    ConvTcDesc g{};
                    g.dt = dt; g.x = pad16; g.C = CP; g.N = Bn; g.H = H; g.W = W; g.ksize = 3; g.stride = 1; g.pad = 1; g.Ho = H; g.Wo = W; g.Cout = C0;
                    g.wmat = wd16_out; g.out_scale = 1.f; g.out = tr->scr_b(); g.mode = TC_MODE_STD; g.stats_cw = tr->m->stats_cw;
                    ConvTcPlan* gp = tr->conv_plan(out_dg_idx, g, &rc);
                    if (!gp) return rc;
                    if ((rc = conv_tc_launch(gp, st))) return rc;
                    tr->launches += 9;
                    tr->tc_wgrads++;
                    return launch_h2f_accumulate(dt, tr->scr_b(), XN.g, (size_t)Bn * H * W * C0, st);
                }
                WgradArgs wa{};
                wa.x1 = XN.d; wa.C1 = C0; wa.N = Bn; wa.H = H; wa.W = W; wa.Cout = Cout; wa.ksize = 3; wa.stride = 1; wa.pad = 1; wa.Ho = H; wa.Wo = W;
                wa.dy = dy4; wa.dy_pitch = 4; wa.dw = gw; wa.scale = 1.f;
                if (gw && (rc = launch_conv_wgrad(wa, st))) return rc;
                tr->launches += 4;
                return launch_conv_dgrad_gather(dy4, 4, pw, Bn, H, W, C0, H, W, Cout, 1, 1, XN.g, st);
            });
        }
        return mo;
    }
};

static int walk(pd_train* t, bool dry, const float* noisy, const float* timesteps, const int64_t* labels, float** mo, float** dm) {
    t->dry = dry;
    t->act_bump = t->aux_bump = 0;
    t->conv_cursor = t->wg_cursor = 0;
    if (dry) { t->scr_max = 0; t->wstage_max = 0; }
    t->tape.clear();
    t->tts.clear();
    t->rc = 0;
    Walk w{t, t->m, t->B};
    *mo = w.forward(noisy, timesteps, labels, dm);
    return t->rc;
}

}  // namespace pd

extern "C" {

int pd_train_create(pd_unet_t* m, int32_t batch, int32_t height, int32_t width, pd_train_t** out) {
    PD_REQUIRE(m && out, "null argument");
    PD_REQUIRE(batch > 0 && height > 0 && width > 0, "bad shape");
    const int ds = 1 << (m->cfg.n_blocks - 1);
    PD_REQUIRE(height % ds == 0 && width % ds == 0, "sample size must be a multiple of 2^(n_blocks-1)");
    PD_REQUIRE(m->cfg.attention_head_dim == 8, "the training step implements attention_head_dim == 8 (the shipped trainable configs)");
    PD_REQUIRE(m->cfg.in_channels <= 4 && m->cfg.out_channels <= 3, "the training step supports in_channels <= 4 and out_channels <= 3");
    for (int i = 0; i < m->cfg.n_blocks; ++i) PD_REQUIRE(m->cfg.block_out_channels[i] % 32 == 0, "block_out_channels must be multiples of 32");
    pd_train* t = new pd_train();
    t->m = m; t->B = batch; t->H = height; t->W = width;
    size_t off = 0;
    for (auto& p : m->params) { t->poff[p.get()] = off; t->poff_by_index.push_back(off); off += p->numel; }
    t->nflat = off;
    float *mo, *dm;
    int rc = walk(t, true, nullptr, nullptr, nullptr, &mo, &dm);
    if (rc) { delete t; return rc; }
    t->act_bytes = t->act_bump;
    t->aux_bytes = t->aux_bump + 2 * t->scr_max + t->wstage_max;
    t->ws_bytes = 2 * t->act_bytes + t->aux_bytes + 1024;
    if (const char* e = getenv("PHENDIFF_B200_TRAIN_TC")) t->tc_mask = (unsigned)atoi(e);
    *out = t;
    return 0;
}

int pd_train_set_precision(pd_train_t* t, int32_t precision) {
    PD_REQUIRE(t, "null argument");
    PD_REQUIRE(precision == PD_PREC_FP32 || precision == PD_PREC_BF16 || precision == PD_PREC_FP16,
               "precision: 0 = fp32 (validation path), 1 = bf16, 2 = fp16 tensor-core operands");
    t->dt = precision == PD_PREC_BF16 ? DT_BF16 : precision == PD_PREC_FP16 ? DT_F16 : DT_F32;
    t->ws = nullptr;   // the workspace plan changes: bind again
    float *mo, *dm;
    int rc = walk(t, true, nullptr, nullptr, nullptr, &mo, &dm);
    if (rc) return rc;
    t->act_bytes = t->act_bump;
    t->aux_bytes = t->aux_bump + 2 * t->scr_max + t->wstage_max;
    t->ws_bytes = 2 * t->act_bytes + t->aux_bytes + 1024;
    return 0;
}

int pd_train_set_loss_scale(pd_train_t* t, const float* scale_dev) {
    PD_REQUIRE(t, "null argument");
    t->loss_scale = scale_dev;
    return 0;
}

int pd_train_tc_counts(pd_train_t* t, int64_t* convs, int64_t* wgrads) {
    PD_REQUIRE(t && convs && wgrads, "null argument");
    *convs = t->tc_convs; *wgrads = t->tc_wgrads;
    return 0;
}

int pd_train_destroy(pd_train_t* t) {
    delete t;
    return 0;
}

int pd_train_num_params_flat(pd_train_t* t, int64_t* numel) {
    PD_REQUIRE(t && numel, "null argument");
    *numel = (int64_t)t->nflat;
    return 0;
}

int pd_train_param_offset(pd_train_t* t, int32_t idx, int64_t* offset) {
    PD_REQUIRE(t && offset && idx >= 0 && idx < (int)t->poff_by_index.size(), "parameter index out of range");
    *offset = (int64_t)t->poff_by_index[idx];
    return 0;
}

int pd_train_workspace_bytes(pd_train_t* t, size_t* bytes) {
    PD_REQUIRE(t && bytes, "null argument");
    *bytes = t->ws_bytes;
    return 0;
}

int pd_train_bind(pd_train_t* t, void* workspace, size_t bytes) {
    PD_REQUIRE(t && workspace, "null argument");
    PD_REQUIRE(bytes >= t->ws_bytes, "workspace too small");
    PD_REQUIRE(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    t->ws = (uint8_t*)workspace;
    return 0;
}

int pd_train_step_grad(pd_train_t* t, const float* params, float* grads, const float* noisy, const float* timesteps, const int64_t* labels,
                       const float* target, const float* sample_weight, float* loss_out, float* model_out, pd_stream_t stream) {
    PD_REQUIRE(t && params && grads && noisy && timesteps && target && loss_out, "null argument");
    PD_REQUIRE(t->ws, "pd_train_bind must be called first");
    int dev = -1;
    PD_CHECK_CUDA(cudaGetDevice(&dev));
    PD_REQUIRE(dev == t->m->device, "the current CUDA device is not the one this handle was created on");
    cudaStream_t s = (cudaStream_t)stream;
    t->P = params; t->G = grads; t->s = s; t->d_input = nullptr; t->forward_pending = false;
    float *mo = nullptr, *dm = nullptr;
    int rc = walk(t, false, noisy, timesteps, labels, &mo, &dm);
    if (rc) return rc;
    PD_REQUIRE(t->act_bump <= t->act_bytes && t->aux_bump + 2 * t->scr_max + t->wstage_max <= t->aux_bytes, "internal: training workspace plan mismatch");
    const size_t per = (size_t)t->m->cfg.out_channels * t->H * t->W;
    if ((rc = launch_mse_loss(mo, target, sample_weight, t->B, per, t->loss_scale, loss_out, dm, s))) return rc;
    if (model_out) PD_CHECK_CUDA(cudaMemcpyAsync(model_out, mo, (size_t)t->B * per * sizeof(float), cudaMemcpyDeviceToDevice, s));
    for (auto it = t->tape.rbegin(); it != t->tape.rend(); ++it)
        if ((rc = (*it)(s))) return rc;
    t->tape.clear();
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

int pd_train_forward(pd_train_t* t, const float* params, const float* x, const float* timesteps, const int64_t* labels, float* model_out,
                     pd_stream_t stream) {
    PD_REQUIRE(t && params && x && timesteps && model_out, "null argument");
    PD_REQUIRE(t->ws, "pd_train_bind must be called first");
    int dev = -1;
    PD_CHECK_CUDA(cudaGetDevice(&dev));
    PD_REQUIRE(dev == t->m->device, "the current CUDA device is not the one this handle was created on");
    cudaStream_t s = (cudaStream_t)stream;
    t->P = params; t->G = nullptr; t->s = s; t->d_input = nullptr; t->forward_pending = false;
    float *mo = nullptr, *dm = nullptr;
    int rc = walk(t, false, x, timesteps, labels, &mo, &dm);
    if (rc) return rc;
    PD_REQUIRE(t->act_bump <= t->act_bytes && t->aux_bump + 2 * t->scr_max + t->wstage_max <= t->aux_bytes, "internal: training workspace plan mismatch");
    const size_t per = (size_t)t->m->cfg.out_channels * t->H * t->W;
    PD_CHECK_CUDA(cudaMemcpyAsync(model_out, mo, (size_t)t->B * per * sizeof(float), cudaMemcpyDeviceToDevice, s));
    t->pending_mo = mo; t->pending_dm = dm; t->forward_pending = true;
    return 0;
}

int pd_train_backward_input(pd_train_t* t, const float* d_model_out, float* d_input, pd_stream_t stream) {
    PD_REQUIRE(t && d_model_out && d_input, "null argument");
    PD_REQUIRE(t->forward_pending, "pd_train_backward_input needs a preceding pd_train_forward on this handle");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t per = (size_t)t->m->cfg.out_channels * t->H * t->W;
    PD_CHECK_CUDA(cudaMemcpyAsync(t->pending_dm, d_model_out, (size_t)t->B * per * sizeof(float), cudaMemcpyDeviceToDevice, s));
    t->d_input = d_input; t->s = s;
    int rc = 0;
    for (auto it = t->tape.rbegin(); it != t->tape.rend(); ++it)
        if ((rc = (*it)(s))) break;
    t->tape.clear();
    t->d_input = nullptr; t->forward_pending = false;
    if (rc) return rc;
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

int pd_guidance_lp_grad(const pd_step_coeffs_t* step, const float* x, const float* model_out, const float* ref, int32_t batch, int64_t per,
                        float p, float* scratch, float* losses, float* d_model_out, float* d_x, pd_stream_t stream) {
    PD_REQUIRE(step && x && model_out && ref && scratch && d_model_out && d_x && batch > 0 && per > 0, "bad argument");
    return launch_guidance_lp_grad(*step, x, model_out, ref, batch, (size_t)per, p, scratch, losses, d_model_out, d_x, (cudaStream_t)stream);
}

int pd_train_launch_count(pd_train_t* t, int64_t* n) {
    PD_REQUIRE(t && n, "null argument");
    *n = t->launches;
    return 0;
}

int pd_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* ema, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int32_t step, float max_grad_norm, float ema_decay, float* scratch,
                  float* grad_norm_out, pd_stream_t stream) {
    PD_REQUIRE(params && grads && exp_avg && exp_avg_sq && scratch && n > 0 && step >= 1, "bad argument");
    return launch_adamw(params, grads, exp_avg, exp_avg_sq, ema, (size_t)n, lr, beta1, beta2, eps, weight_decay, step, max_grad_norm, ema_decay,
                        scratch, grad_norm_out, (cudaStream_t)stream);
}

int pd_adamw_step_scaled(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* ema, int64_t n, float lr, float beta1,
                         float beta2, float eps, float weight_decay, float max_grad_norm, float ema_decay, pd_grad_scaler_state_t* state,
                         float growth_factor, float backoff_factor, int32_t growth_interval, float* scratch, float* grad_norm_out,
                         pd_stream_t stream) {
    PD_REQUIRE(params && grads && exp_avg && exp_avg_sq && state && scratch && n > 0, "bad argument");
    PD_REQUIRE(growth_factor > 1.f && backoff_factor > 0.f && backoff_factor < 1.f && growth_interval >= 1,
               "grad scaler: growth_factor > 1, 0 < backoff_factor < 1 and growth_interval >= 1 (torch.amp.GradScaler's conditions)");
    return launch_adamw_scaled(params, grads, exp_avg, exp_avg_sq, ema, (size_t)n, lr, beta1, beta2, eps, weight_decay, max_grad_norm, ema_decay,
                               state, growth_factor, backoff_factor, growth_interval, scratch, grad_norm_out, (cudaStream_t)stream);
}

}  // extern "C"
