// eh_plan.cu -- the planner of libeasyhybrid_cuda.so: eh_model_desc -> kernel variant + layout tables (host code only).
//
// Which path serves a model (specialised exact-fp32 variant / generic exact-fp32 variant with an interpreted or run-time
// compiled process model / bf16 tcgen05 path), how several Dense chains are embedded block-diagonally into one chain
// (MultiNNHybridModel, src/models/GenericHybridModel.jl:169-189; chains of unequal depth on pass-through units), the
// reference's flat ComponentArray layout (a15) and the gather / scatter tables between it and the kernels' images.
#include "eh_ctx.h"

namespace eh {
namespace rt {
namespace {
// Plan for the tensor-core path: one or several Dense chains embedded block-diagonally into one padded chain
// (eh_wide_kernels.cuh, WideDims).  Fills the parts of the ctx the shared host code reads (record layout, slots, loss,
// optimiser) and the WideModel handed to WideNet::create.  Chains that differ in depth or activation (2..6 hidden layers)
// take the per-unit form: a shallower chain carries its last hidden layer up to layer NH on pass-through units (weight 1
// from the unit below, bias 0, identity activation: exact in bf16), and every hidden unit has its own activation.
eh_status build_plan_wide(eh_ctx* c, const eh_model_desc* d, bool is_prog)
{
    const int NC = d->n_chains;
    const eh_chain_desc& c0 = d->chains[0];
    int NH = 0;
    for (int k = 0; k < NC; k++) NH = std::max(NH, d->chains[k].n_hidden);
    int P = 0, NOUT = 0, wl[8] = {0};
    bool per_unit = false, per_unit_ok = true;
    for (int k = 0; k < NC; k++) {
        const eh_chain_desc& ch = d->chains[k];
        if ((ch.input_batchnorm != 0) != (c0.input_batchnorm != 0))
            return fail(c, EH_EUNSUPPORTED, "chains of one model must share input_batchnorm on the tensor-core path");
        if (ch.n_in < 1 || ch.n_out < 1) return fail(c, EH_EINVAL, "chain %d: n_in / n_out must be positive", k);
        per_unit |= ch.n_hidden != NH || ch.activation != c0.activation;
        per_unit_ok &= ch.activation == EH_ACT_TANH || ch.activation == EH_ACT_SIGMOID || ch.activation == EH_ACT_RELU ||
                       ch.activation == EH_ACT_IDENTITY;
        P += ch.n_in;
        NOUT += ch.n_out;
        for (int l = 0; l < ch.n_hidden && l < 8; l++)
            if (ch.hidden[l] < 1) return fail(c, EH_EINVAL, "chain %d: hidden width must be positive", k);
        for (int l = 0; l < NH && l < 8; l++) wl[l] += ch.hidden[std::min(l, ch.n_hidden - 1)];   // (pass-through units too)
    }
    int hmax = 0;
    for (int l = 0; l < NH && l < 8; l++) hmax = std::max(hmax, wl[l]);
    if (NH > 7 || !eh::wide::WideNet::supported(P, hmax, NH, NOUT, c0.activation, d->process_model) ||
        (per_unit && (NH < 2 || !per_unit_ok)))
        return fail(c, EH_EUNSUPPORTED,
                    "no fused kernel for this model: the register-tile kernels serve 1..3 hidden layers of summed width <= 32 "
                    "(all activations, <= 8 inputs, <= 2 outputs); the wide path serves 1..4 chains with one input_batchnorm "
                    "setting and <= 12 inputs and <= 4 outputs in total (more than 8 / 2 only with some layer wider than 32; "
                    "3..4 outputs: traced process models): one hidden layer of summed width 33..512 (exact fp32, all "
                    "activations, one activation for all chains) or 2..6 hidden layers of summed width <= 512 per layer, "
                    "pass-through units of shallower chains included (bf16 tensor cores, tanh / sigmoid / relu; chains may "
                    "differ in depth and activation) "
                    "(got process_model=%d chains=%d inputs=%d hidden=%d x (<= %d) outputs=%d activation=%d)",
                    d->process_model, NC, P, NH, hmax, NOUT, c0.activation);
    // (one hidden layer: the fused exact-fp32 kernel k_wide_one, images padded to a multiple of 64 units)
    const int HP = NH == 1 ? eh::wide::WideNet::one_width(hmax) : eh::wide::WideNet::padded_width(hmax);
    Variant& wv = c->wide_var;
    memset(&wv, 0, sizeof wv);
    wv.pm = d->process_model; wv.P = P; wv.NH = NH; wv.H = HP; wv.NOUT = NOUT; wv.act = c0.activation;
    wv.scale = d->scale_nn_outputs ? 1 : 0;
    wv.engine = 3; wv.chunk = 128;
    wv.F = is_prog ? d->n_forc : 1; wv.NPS = is_prog ? d->n_params : 2;
    wv.T = is_prog ? d->n_targ : ((d->process_model == EH_PM_LINEAR2 || d->process_model == EH_PM_EXPO2) ? 2 : 1);
    wv.R4 = rup4(wv.P + wv.F + wv.T);
    wv.NW = 0; wv.NPART = NSTAT; wv.off_stats = 0; wv.stage_floats = NSTAT; wv.max_warps = 8;
    wv.name = NH == 1 ? "wide/fp32-one-hidden" : per_unit ? "wide/bf16-tcgen05-per-unit" : "wide/bf16-tcgen05";
    if (wv.T != d->n_targ) return fail(c, EH_EINVAL, "process model yields %d targets, descriptor has %d", wv.T, d->n_targ);
    const Variant* v = &wv;
    c->var = v; c->var2 = nullptr;
    c->n_pred_raw = d->n_pred; c->n_forc_raw = d->n_forc; c->n_targ = d->n_targ;
    c->use_bn = c0.input_batchnorm ? 1 : 0;
    c->real_in = P;
    c->n_chains = NC;
    for (int k = 0, o = 0; k < NC && k < 4; k++) { c->chain_in0[k] = o; c->chain_nin[k] = d->chains[k].n_in; o += d->chains[k].n_in; }
    c->flags = (unsigned)d->flags;
    c->persist_ok = false;
    c->pm_id = d->process_model;

    // flat layout (reference ComponentArray order): chain after chain, per layer W (out x in, column-major) then b; then phi.
    // Embedding: chain k owns units [uoff[l], uoff[l] + h) of hidden layer l, inputs [ioff, ioff + n_in), outputs [ooff, ..);
    // a chain of depth dk < NH owns its pass-through units in layers dk + 1 .. NH, and its output layer reads those of NH
    c->h_wmap.assign((size_t)0, 0);
    eh::wide::WideModel& wm = c->wide_model;
    memset(&wm, 0, sizeof wm);
    wm.per_unit = per_unit ? 1 : 0;
    memset(wm.uact, EH_ACT_IDENTITY, sizeof wm.uact);
    int off = 0, ioff = 0, ooff = 0, uoff[8] = {0};
    std::vector<int> out_row0((size_t)NC, 0);
    std::vector<std::pair<int, int>> wranges;   // (flat offset, count) of every Dense weight matrix, with its chain in l2_chain
    std::vector<int> l2_chain;
    auto push = [&](int kind, int l, int r, int cc) { c->h_wmap.push_back(kind); c->h_wmap.push_back(l); c->h_wmap.push_back(r); c->h_wmap.push_back(cc); };
    for (int k = 0; k < NC; k++) {
        const eh_chain_desc& ch = d->chains[k];
        const int dk = ch.n_hidden;
        out_row0[k] = ooff;
        for (int l = 1; l <= dk + 1; l++) {
            const bool outl = l == dk + 1;
            const int hout = outl ? ch.n_out : ch.hidden[l - 1];
            const int hin = l == 1 ? ch.n_in : ch.hidden[l - 2];
            const int ro = outl ? ooff : uoff[l - 1];                        // image row origin (output units)
            const int co = l == 1 ? ioff : uoff[outl ? NH - 1 : l - 2];      // image column origin (input units)
            const int li = outl ? NH + 1 : l;                                // layer of the embedded chain
            if (!outl && l >= 2) {
                if (wm.n_blocks >= 32) return fail(c, EH_EUNSUPPORTED, "too many weight blocks");
                auto& bk = wm.blocks[wm.n_blocks++];
                bk.l = l; bk.flat_off = off; bk.hout = hout; bk.hin = hin; bk.o_off = ro; bk.i_off = co;
            }
            const int kind = l == 1 ? eh::wide::WK_W1 : (outl ? eh::wide::WK_WO : eh::wide::WK_WH);
            for (int i = 0; i < hin; i++)
                for (int o = 0; o < hout; o++) push(kind, li, ro + o, co + i);
            wranges.push_back({off, hout * hin});
            l2_chain.push_back(k);
            off += hout * hin;
            for (int o = 0; o < hout; o++) push(outl ? eh::wide::WK_BO : eh::wide::WK_B, li, ro + o, 0);
            off += hout;
        }
        for (int l = 1; l <= NH && l <= 6; l++) {
            const int w = ch.hidden[std::min(l, dk) - 1];
            memset(&wm.uact[l - 1][uoff[l - 1]], l <= dk ? ch.activation : (int)EH_ACT_IDENTITY, (size_t)w);
            if (l > dk) {   // pass-through run: unit j of layer l - 1 -> unit j of layer l
                if (wm.n_pass >= 24) return fail(c, EH_EUNSUPPORTED, "too many pass-through runs");
                auto& pr = wm.pass[wm.n_pass++];
                pr.l = l; pr.r0 = uoff[l - 1]; pr.c0 = uoff[l - 2]; pr.n = w;
            }
        }
        for (int l = 0; l < NH; l++) uoff[l] += ch.hidden[std::min(l, dk - 1)];
        ioff += ch.n_in;
        ooff += ch.n_out;
    }
    c->ntheta = off;
    int ng = 0;
    for (int p = 0; p < d->n_params; p++)
        if (d->role[p] == EH_ROLE_GLOBAL) ng = std::max(ng, d->role_index[p] + 1);
    c->nglob = ng;
    c->nflat = off + ng;
    for (int g = 0; g < ng; g++) push(eh::wide::WK_PHI, 0, g, 0);
    c->h_wsrc.assign((size_t)ng, -1);
    for (int g = 0; g < ng; g++) c->h_wsrc[(size_t)g] = off + g;
    c->h_pmap.assign((size_t)c->nflat, 0);
    c->h_pspan.assign((size_t)c->nflat, 0.f);
    c->h_cells.assign((size_t)2 * c->nflat, -1);

    // canonical slots: built-in forms bind (param, param, forcing); traced programs address the parameter table directly
    c->nparam_desc = d->n_params;
    c->slot_of_param.assign((size_t)d->n_params, -1);
    memset(c->slots, 0, sizeof c->slots);
    for (int s = 0; s < MAXPS; s++) c->slots[s].role = ROLE_FIXED;
    for (int s = 0; s < v->NPS; s++) {
        const int pi = is_prog ? s : d->pm_args[s].index;
        if (pi < 0 || pi >= d->n_params) return fail(c, EH_EINVAL, "pm_args[%d].index out of range", s);
        PSlot& sl = c->slots[s];
        sl.role = d->role[pi];
        sl.lo = d->lower[pi];
        sl.span = d->upper[pi] - d->lower[pi];
        sl.fixedv = d->deflt[pi];
        if (sl.role == EH_ROLE_NEURAL) {
            const int chain = d->role_index[pi] >> 16, row = d->role_index[pi] & 0xffff;
            if (chain < 0 || chain >= NC || row >= d->chains[chain].n_out)
                return fail(c, EH_EINVAL, "neural parameter %d refers to chain %d row %d", pi, chain, row);
            sl.idx = out_row0[(size_t)chain] + row;
        } else if (sl.role == EH_ROLE_GLOBAL) {
            sl.idx = d->role_index[pi];
        }
        c->slot_of_param[pi] = s;
    }
    for (int i = 0; i < 4; i++) c->pmc[i] = d->pm_consts[i];
    c->h_slot_of_flat.assign((size_t)c->nflat, -1);
    for (int g = 0; g < ng; g++)
        for (int s = 0; s < v->NPS; s++)
            if (c->slots[s].role == ROLE_GLOBAL && c->slots[s].idx == g) c->h_slot_of_flat[(size_t)off + g] = s;

    // record columns: the chains' inputs one after the other, forcing(s), targets
    c->ncols = 0;
    for (int k = 0; k < NC; k++)
        for (int q = 0; q < d->chains[k].n_in; q++) {
            const int col = d->chains[k].in_cols[q];
            if (col < 0 || col >= d->n_pred) return fail(c, EH_EINVAL, "chain %d in_cols[%d] out of range", k, q);
            c->src_kind[c->ncols] = 0; c->src_idx[c->ncols] = col; c->ncols++;
        }
    if (is_prog) {
        for (int fi = 0; fi < d->n_forc; fi++) { c->src_kind[c->ncols] = 1; c->src_idx[c->ncols] = fi; c->ncols++; }
    } else {
        const int fi = d->pm_args[2].index;
        if (fi < 0 || fi >= d->n_forc) return fail(c, EH_EINVAL, "forcing index out of range");
        c->src_kind[c->ncols] = 1; c->src_idx[c->ncols] = fi; c->ncols++;
    }
    for (int t = 0; t < d->n_targ; t++) { c->src_kind[c->ncols] = 1; c->src_idx[c->ncols] = d->n_forc + t; c->ncols++; }

    // loss / optimiser.  rmse over several targets and pearsonLoss / kgeLoss / pbkgeLoss need statistics of the batch's
    // predictions before the seeds exist: those targets run as LOSS_AFFINE behind a statistics pass of the head kernel
    // (WideNet::step); single-target rmse keeps LOSS_RMSE and its 1 / (2 rmse) factor
    for (int t = 0; t < d->n_targ; t++) {
        const int lk = d->loss_per_target[t];
        if (lk < 0 || lk > EH_LOSS_PBKGELOSS) return fail(c, EH_EINVAL, "loss_per_target[%d]=%d unknown", t, lk);
        c->loss_kind_abi[t] = lk;
        const bool stat = lk >= EH_LOSS_PEARSONLOSS || (lk == EH_LOSS_RMSE && d->n_targ > 1);
        c->loss_kind[t] = stat ? (int)LOSS_AFFINE : lk;
        c->stat_loss |= stat;
    }
    // native extra loss lambda * weight_l2(ps.<chains>; normalize) (ABI version 2), as on the exact-fp32 path: 2 lambda [/ n]
    // on the Dense weight entries of the selected chains (every layer, output layer included), 0 elsewhere
    c->l2_on = d->abi_version >= 2 && d->l2_lambda != 0.f;
    if (c->l2_on) {
        auto picked = [&](int k) { return !d->l2_chain_mask || ((d->l2_chain_mask >> k) & 1u); };
        long long nw = 0;
        for (size_t i = 0; i < wranges.size(); i++) nw += picked(l2_chain[i]) ? wranges[i].second : 0;
        const double lam = (double)d->l2_lambda / ((d->l2_normalize && nw > 0) ? (double)nw : 1.0);
        c->l2_aggw = d->agg == EH_AGG_MEAN ? 0.5f : 1.0f;
        c->l2_loss_coef = (float)lam;
        c->h_l2coef.assign((size_t)c->nflat, 0.f);
        for (size_t i = 0; i < wranges.size(); i++)
            for (int j = 0; picked(l2_chain[i]) && j < wranges[i].second; j++) c->h_l2coef[(size_t)wranges[i].first + j] = (float)(2.0 * lam);
    }
    c->agg_mean = d->agg == EH_AGG_MEAN;
    c->opt_kind = d->opt_kind;
    if (c->opt_kind < 0 || c->opt_kind > 3) return fail(c, EH_EINVAL, "opt_kind=%d unknown", d->opt_kind);
    c->adamw_coupled = d->adamw_decay_coupled_eta;
    c->eta = d->eta; c->beta1 = d->beta1; c->beta2 = d->beta2; c->eps = d->eps; c->lambda = d->lambda;
    c->bn_mean.assign((size_t)P, 0.f);
    c->bn_var.assign((size_t)P, 1.f);

    wm.P = P; wm.H = HP; wm.NH = NH; wm.NOUT = NOUT; wm.R4 = v->R4; wm.nflat = c->nflat; wm.ntheta = c->ntheta;
    wm.h_map = c->h_wmap.data();
    wm.act = c0.activation; wm.scale = d->scale_nn_outputs ? 1 : 0; wm.pm = d->process_model;
    wm.T = v->T; wm.F = v->F; wm.NPS = v->NPS; wm.use_bn = c->use_bn; wm.agg_mean = c->agg_mean;
    for (int t = 0; t < MAXT; t++) { wm.loss_kind[t] = c->loss_kind[t]; wm.loss_kind_abi[t] = c->loss_kind_abi[t]; }
    wm.l2_aggw = c->l2_aggw; wm.l2_loss_coef = c->l2_loss_coef;   // (d_l2coef: set when the device copy exists)
    for (int s2 = 0; s2 < MAXPS; s2++) {
        wm.slot[s2].role = c->slots[s2].role; wm.slot[s2].idx = c->slots[s2].idx; wm.slot[s2].lo = c->slots[s2].lo;
        wm.slot[s2].span = c->slots[s2].span; wm.slot[s2].fixedv = c->slots[s2].fixedv;
    }
    for (int i = 0; i < 4; i++) wm.pmc[i] = c->pmc[i];
    wm.opt_kind = c->opt_kind; wm.adamw_coupled = c->adamw_coupled;
    wm.eta = c->eta; wm.beta1 = c->beta1; wm.beta2 = c->beta2; wm.eps = c->eps; wm.lambda = c->lambda;
    wm.nsm = c->nsm;
    if (is_prog) {
        wm.prog_len = d->pm_len;
        for (int i = 0; i < d->pm_len; i++) {
            wm.prog_op[i] = (short)d->pm_prog[i].op; wm.prog_a[i] = (short)d->pm_prog[i].a; wm.prog_b[i] = (short)d->pm_prog[i].b;
            wm.prog_imm[i] = d->pm_prog[i].imm;
        }
        for (int t = 0; t < d->n_targ; t++) wm.prog_out[t] = d->pm_outputs[t];
    }
    return EH_OK;
}

// The process model as a straight-line program for the generic variants: a traced one is taken as it is (already
// validated), a built-in form is written out from its (param, param, forcing) binding -- PARAM operands address the
// descriptor's parameter table, FORCING operands its forcing columns, like traced programs do.
bool builtin_as_program(const eh_model_desc* d, bool is_prog, std::vector<eh_pm_instr>& prog, std::vector<int>& out)
{
    prog.clear();
    out.clear();
    if (is_prog) {
        prog.assign(d->pm_prog, d->pm_prog + d->pm_len);
        out.assign(d->pm_outputs, d->pm_outputs + d->n_targ);
        return true;
    }
    auto emit = [&](int op, int a, int b, float imm) {
        eh_pm_instr in;
        memset(&in, 0, sizeof in);
        in.op = op; in.a = a; in.b = b; in.imm = imm;
        prog.push_back(in);
        return (int)prog.size() - 1;
    };
    const int pa = emit(EH_OP_PARAM, d->pm_args[0].index, 0, 0.f);
    const int pb = emit(EH_OP_PARAM, d->pm_args[1].index, 0, 0.f);
    const int f = emit(EH_OP_FORCING, d->pm_args[2].index, 0, 0.f);
    switch (d->process_model) {
    case EH_PM_RBQ10: {   // rb * Q10^(0.1 (ta - tref))
        const int tref = emit(EH_OP_CONST, 0, 0, d->pm_consts[0]);
        const int dt = emit(EH_OP_SUB, f, tref, 0.f);
        const int tenth = emit(EH_OP_CONST, 0, 0, 0.1f);
        const int e = emit(EH_OP_MUL, tenth, dt, 0.f);
        const int pw = emit(EH_OP_POW, pb, e, 0.f);
        out.push_back(emit(EH_OP_MUL, pa, pw, 0.f));
        break;
    }
    case EH_PM_EXPO:
    case EH_PM_EXPO2: {   // Resp0 * exp(k T) (; twice that)
        const int kt = emit(EH_OP_MUL, pb, f, 0.f);
        const int ex = emit(EH_OP_EXP, kt, 0, 0.f);
        const int y0 = emit(EH_OP_MUL, pa, ex, 0.f);
        out.push_back(y0);
        if (d->process_model == EH_PM_EXPO2) {
            const int two = emit(EH_OP_CONST, 0, 0, 2.f);
            out.push_back(emit(EH_OP_MUL, two, y0, 0.f));
        }
        break;
    }
    case EH_PM_LINEAR:
    case EH_PM_LINEAR2: {   // a x + b (; 2 a x + b)
        const int ax = emit(EH_OP_MUL, pa, f, 0.f);
        out.push_back(emit(EH_OP_ADD, ax, pb, 0.f));
        if (d->process_model == EH_PM_LINEAR2) {
            const int two = emit(EH_OP_CONST, 0, 0, 2.f);
            const int ax2 = emit(EH_OP_MUL, two, ax, 0.f);
            out.push_back(emit(EH_OP_ADD, ax2, pb, 0.f));
        }
        break;
    }
    default:
        return false;
    }
    if ((int)out.size() != d->n_targ) return false;
    for (int k = 0; k < 3; k++) {
        const int lim = k < 2 ? d->n_params : d->n_forc;
        if (d->pm_args[k].index < 0 || d->pm_args[k].index >= lim) return false;
    }
    return true;
}


// ---- traced program -> built-in form ---------------------------------------------------------------------------------
// A host that traces the user's mechanistic_model (GenericHybridModel.jl:425 takes any callable) hands over a program.
// If that program IS one of the built-in forms -- up to the order of commutative operands and the binding of
// (parameter, parameter, forcing) -- the specialised kernels serve it: the comparison is done here, once, so every host
// (Julia shim, Python mirror, C harness) gets the same path selection.  Canonical string of an expression: commutative
// operands sorted; constants by their float32 bit pattern.
static std::string pm_canon(const eh_pm_instr* prog, int vid)
{
    const eh_pm_instr& in = prog[vid];
    char buf[48];
    switch (in.op) {
    case EH_OP_CONST: { unsigned u; memcpy(&u, &in.imm, 4); snprintf(buf, sizeof buf, "c%08x", u); return buf; }
    case EH_OP_FORCING: snprintf(buf, sizeof buf, "F%d", in.a); return buf;
    case EH_OP_PARAM: snprintf(buf, sizeof buf, "P%d", in.a); return buf;
    default: break;
    }
    if (in.op >= EH_OP_NEG) return "u" + std::to_string(in.op) + "(" + pm_canon(prog, in.a) + ")";
    std::string a = pm_canon(prog, in.a), b = pm_canon(prog, in.b);
    const bool comm = in.op == EH_OP_ADD || in.op == EH_OP_MUL || in.op == EH_OP_MIN || in.op == EH_OP_MAX;
    if (comm && b < a) std::swap(a, b);
    return "b" + std::to_string(in.op) + "(" + a + "," + b + ")";
}

// the built-in forms written as programs over (param pi, param pj, forcing fk, const c0); returns the output value ids
static int builtin_form_program(int pm, int pi, int pj, int fk, float c0, std::vector<eh_pm_instr>& p, int out[2])
{
    auto emit = [&](int op, int a, int b, float imm) { p.push_back(eh_pm_instr{op, a, b, imm}); return (int)p.size() - 1; };
    const int P0 = emit(EH_OP_PARAM, pi, 0, 0.f), P1 = emit(EH_OP_PARAM, pj, 0, 0.f), F0 = emit(EH_OP_FORCING, fk, 0, 0.f);
    switch (pm) {
    case EH_PM_RBQ10: {   // p0 * p1 ^ (0.1 (f0 - c0))
        const int d = emit(EH_OP_SUB, F0, emit(EH_OP_CONST, 0, 0, c0), 0.f);
        const int e = emit(EH_OP_MUL, emit(EH_OP_CONST, 0, 0, 0.1f), d, 0.f);
        out[0] = emit(EH_OP_MUL, P0, emit(EH_OP_POW, P1, e, 0.f), 0.f);
        return 1;
    }
    case EH_PM_EXPO: out[0] = emit(EH_OP_MUL, P0, emit(EH_OP_EXP, emit(EH_OP_MUL, P1, F0, 0.f), 0, 0.f), 0.f); return 1;
    case EH_PM_LINEAR: out[0] = emit(EH_OP_ADD, emit(EH_OP_MUL, P0, F0, 0.f), P1, 0.f); return 1;
    case EH_PM_LINEAR2: {
        out[0] = emit(EH_OP_ADD, emit(EH_OP_MUL, P0, F0, 0.f), P1, 0.f);
        const int twoa = emit(EH_OP_MUL, emit(EH_OP_CONST, 0, 0, 2.f), P0, 0.f);
        out[1] = emit(EH_OP_ADD, emit(EH_OP_MUL, twoa, F0, 0.f), P1, 0.f);
        return 2;
    }
    case EH_PM_EXPO2: {
        out[0] = emit(EH_OP_MUL, P0, emit(EH_OP_EXP, emit(EH_OP_MUL, P1, F0, 0.f), 0, 0.f), 0.f);
        out[1] = emit(EH_OP_MUL, emit(EH_OP_CONST, 0, 0, 2.f), out[0], 0.f);
        return 2;
    }
    default: return 0;
    }
}

// true: the (validated) program of `d` equals built-in form *pm with the binding args[3] and constant consts[0]
static bool match_builtin_program(const eh_model_desc* d, int* pm, eh_pm_arg args[3], float consts[4])
{
    std::vector<std::string> want;
    for (int t = 0; t < d->n_targ; t++) want.push_back(pm_canon(d->pm_prog, d->pm_outputs[t]));
    std::vector<float> cs;
    for (int i = 0; i < d->pm_len; i++)
        if (d->pm_prog[i].op == EH_OP_CONST) cs.push_back(d->pm_prog[i].imm);
    const int forms[] = {EH_PM_RBQ10, EH_PM_EXPO, EH_PM_LINEAR, EH_PM_LINEAR2, EH_PM_EXPO2};
    for (int form : forms)
        for (int pi = 0; pi < d->n_params; pi++)
            for (int pj = 0; pj < d->n_params; pj++) {
                if (pi == pj) continue;
                for (int fk = 0; fk < d->n_forc; fk++) {
                    std::vector<float> trial = form == EH_PM_RBQ10 ? cs : std::vector<float>{0.f};
                    for (float c0 : trial) {
                        std::vector<eh_pm_instr> p;
                        int out[2] = {0, 0};
                        if (builtin_form_program(form, pi, pj, fk, c0, p, out) != d->n_targ) continue;
                        bool same = true;
                        for (int t = 0; t < d->n_targ && same; t++) same = pm_canon(p.data(), out[t]) == want[(size_t)t];
                        if (same) {
                            *pm = form;
                            args[0] = eh_pm_arg{0, pi}; args[1] = eh_pm_arg{0, pj}; args[2] = eh_pm_arg{1, fk};
                            consts[0] = c0; consts[1] = consts[2] = consts[3] = 0.f;
                            return true;
                        }
                    }
                }
            }
    return false;
}


}  // namespace

eh_status build_plan(eh_ctx* c, const eh_model_desc* d)
{
    // (version 1 descriptors end before the weight_l2 fields: those are only read from version >= 2)
    if (d->abi_version < 1 || d->abi_version > EH_ABI_VERSION) return fail(c, EH_EINVAL, "abi_version %d not in 1..%d", d->abi_version, EH_ABI_VERSION);
    if (d->n_targ < 1 || d->n_targ > MAXT) return fail(c, EH_EUNSUPPORTED, "n_targ=%d not in 1..%d", d->n_targ, MAXT);
    if (d->n_chains < 1 || d->n_chains > 4) return fail(c, EH_EUNSUPPORTED, "n_chains=%d not in 1..4", d->n_chains);
    const bool is_prog = d->process_model == EH_PM_PROGRAM;
    if (is_prog) {
        // a traced process model: validated here, interpreted per sample by the tensor-core path's head kernel
        if (d->pm_len < 1 || d->pm_len > PM_MAXLEN || !d->pm_prog || !d->pm_outputs)
            return fail(c, EH_EUNSUPPORTED, "traced process model: 1..%d instructions supported (got %d)", PM_MAXLEN, d->pm_len);
        if (d->n_params < 1 || d->n_params > MAXPS || d->n_forc < 0 || d->n_forc > 4 || d->n_targ > 2)
            return fail(c, EH_EUNSUPPORTED, "traced process model: <= %d parameters, <= 4 forcings, <= 2 targets", MAXPS);
        for (int i = 0; i < d->pm_len; i++) {
            const eh_pm_instr& in = d->pm_prog[i];
            const bool leaf = in.op == EH_OP_CONST || in.op == EH_OP_FORCING || in.op == EH_OP_PARAM;
            const bool binary = in.op >= EH_OP_ADD && in.op <= EH_OP_MAX, unary = in.op >= EH_OP_NEG && in.op <= EH_OP_COS;
            if (!leaf && !binary && !unary) return fail(c, EH_EINVAL, "pm_prog[%d]: unknown op %d", i, in.op);
            if (in.op == EH_OP_FORCING && (in.a < 0 || in.a >= d->n_forc)) return fail(c, EH_EINVAL, "pm_prog[%d]: forcing %d out of range", i, in.a);
            if (in.op == EH_OP_PARAM && (in.a < 0 || in.a >= d->n_params)) return fail(c, EH_EINVAL, "pm_prog[%d]: parameter %d out of range", i, in.a);
            if ((binary || unary) && (in.a < 0 || in.a >= i)) return fail(c, EH_EINVAL, "pm_prog[%d]: operand a=%d is not an earlier value", i, in.a);
            if (binary && (in.b < 0 || in.b >= i)) return fail(c, EH_EINVAL, "pm_prog[%d]: operand b=%d is not an earlier value", i, in.b);
        }
        for (int t = 0; t < d->n_targ; t++)
            if (d->pm_outputs[t] < 0 || d->pm_outputs[t] >= d->pm_len) return fail(c, EH_EINVAL, "pm_outputs[%d] out of range", t);
        // a traced program that IS a built-in form takes the specialised kernels (EH_NO_PM_MATCH=1: keep it as a program)
        int pm_id = 0;
        eh_pm_arg margs[3];
        float mconsts[4];
        if (!getenv("EH_NO_PM_MATCH") && match_builtin_program(d, &pm_id, margs, mconsts)) {
            eh_model_desc dd = *d;
            dd.process_model = pm_id; dd.n_pm_args = 3; dd.pm_args = margs;
            for (int i = 0; i < 4; i++) dd.pm_consts[i] = mconsts[i];
            dd.pm_prog = nullptr; dd.pm_len = 0; dd.pm_outputs = nullptr;
            return build_plan(c, &dd);
        }
    }
    const eh_chain_desc& ch = d->chains[0];
    const int NC = d->n_chains;
    // several chains (MultiNNHybridModel, GenericHybridModel.jl:169-189, 458-530) are embedded block-diagonally into ONE
    // chain: chain k owns a range of the inputs, of the units of every hidden layer and of the outputs; weights between
    // units of different chains do not exist (zero cells of the image that no flat entry feeds).  Totals per level:
    // Chains of different depth (hidden sizes differ per parameter, GenericHybridModel.jl:169-189): the embedded chain
    // has the depth of the deepest one; a shallower chain carries its last hidden layer forward through pass-through
    // units (weight 1 from the unit below, no bias, identity activation -- cells fed by no flat entry) up to the common
    // output layer.  The generic variants know pass-through units, and so does the tensor-core path (build_plan_wide) once
    // some layer is wider than 32 units.
    int Pt = 0, Ot = 0, wsum[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    bool uniform = true, same_depth = true, same_act = true, any_swish = false;
    int NHmax = 0;
    for (int k = 0; k < NC; k++) NHmax = std::max(NHmax, d->chains[k].n_hidden);
    for (int k = 0; k < NC; k++) {
        const eh_chain_desc& ck = d->chains[k];
        if (ck.n_in < 1) return fail(c, EH_EINVAL, "chain %d has no inputs", k);
        if (ck.n_hidden < 1) return fail(c, EH_EINVAL, "chain needs at least one hidden layer");
        if (ck.input_batchnorm != ch.input_batchnorm) uniform = false;
        if (ck.activation != ch.activation) same_act = false;
        if (ck.activation == EH_ACT_SWISH) any_swish = true;
        if (ck.n_hidden != NHmax) same_depth = false;
        Pt += ck.n_in; Ot += ck.n_out;
        for (int l = 0; l < NHmax && l < 8; l++) wsum[l] += ck.hidden[std::min(l, ck.n_hidden - 1)];
    }
    if (NC == 1 && ch.n_in > MAXP) return fail(c, EH_EUNSUPPORTED, "chain n_in=%d not in 1..%d", ch.n_in, MAXP);
    int hmax = 0;
    for (int l = 0; l < NHmax && l < 8; l++) hmax = std::max(hmax, wsum[l]);
    if (!is_prog && (d->n_pm_args != 3 || d->pm_args[0].kind != 0 || d->pm_args[1].kind != 0 || d->pm_args[2].kind != 1))
        return fail(c, EH_EINVAL, "built-in process models take (param, param, forcing) arguments");
    // Which path?  The exact-fp32 register-tile kernels exist for one to three hidden layers of width <= 32; every other chain
    // (wider or deeper, up to 6 hidden layers of up to 512 units, padded to 256 / 512 internally) runs on the bf16
    // tcgen05 GEMM path.
    const bool wide = false;   // (this function continues with the register-tile plan only)
    const int scale_flag = d->scale_nn_outputs ? 1 : 0;
    // (the register-tile kernels keep theta / m / v in shared memory and update them in one CTA: <= 2048 - NSTAT entries)
    long long nflat_est = 0;
    for (int k = 0; k < NC; k++) {
        const eh_chain_desc& ck = d->chains[k];
        int prev = ck.n_in;
        for (int l = 0; l < ck.n_hidden; l++) { nflat_est += (long long)(prev + 1) * ck.hidden[l]; prev = ck.hidden[l]; }
        nflat_est += (long long)(prev + 1) * ck.n_out;
    }
    for (int p = 0; p < d->n_params; p++)
        if (d->role[p] == EH_ROLE_GLOBAL) nflat_est++;
    const bool small_shape = uniform && NHmax <= 3 && hmax <= 32 && nflat_est <= 2048 - NSTAT;
    const Variant* v = nullptr;
    // 1. a specialised variant of a built-in form (the BASELINE configurations); engine 1 (tensor pipe, 3xTF32) on
    //    request where one exists, engine 0 (exact-fp32 FFMA2) otherwise
    if (small_shape && !is_prog && NC == 1) {
        if (d->flags & EH_FLAG_TENSOR_PIPE)
            v = find_variant(d->process_model, ch.n_in, ch.n_hidden, rup4(hmax), ch.n_out, ch.activation, scale_flag, 1);
        if (!v) v = find_variant(d->process_model, ch.n_in, ch.n_hidden, rup4(hmax), ch.n_out, ch.activation, scale_flag, 0);
    }
    // 2. the generic exact-fp32 variants: the process model (a traced one, or a built-in form without a specialised
    //    variant, rewritten as a program) is interpreted per sample -- value and reverse sweep -- inside the same
    //    register-tile kernels; chain inputs are padded up to the compiled count (2 / 4 / 8) with zero columns,
    //    scale_nn_outputs is a run-time flag.  EH_NO_SMALL_PROGRAM=1 sends these models to the tensor-core path.
    std::vector<eh_pm_instr> prog;
    std::vector<int> prog_out;
    bool use_prog = false, auto_jit = false;
    PmProgData pd;
    unsigned char unit_act[3][32];
    // run-time specialisation of the traced program (EH_FLAG_JIT, or EH_JIT=1 for every traced model; EH_JIT=0: never)
    const char* env_jit = getenv("EH_JIT");
    const bool want_jit = env_jit ? (env_jit[0] && env_jit[0] != '0') : (d->flags & EH_FLAG_JIT) != 0;
    if (!v && small_shape && !getenv("EH_NO_SMALL_PROGRAM") && d->n_params >= 1 && d->n_params <= MAXPS && d->n_forc <= PmProgram::NF &&
        d->n_targ <= PmProgram::NT) {
        // (with run-time compilation the tightest shape that holds the model is taken -- inputs padded to 2 / 4 / 8 / 12,
        // width 8 / 16 / 24 / 32, up to four chain outputs; the compiled-in variants know 2 / 4 / 8 inputs, width 16 / 32 and
        // one or two outputs)
        // chains that differ in activation (an activation per parameter, GenericHybridModel.jl:168-174): every unit gets its
        // own activation in the generated code; the shape's activation is only the container (swish if any chain uses it:
        // its sigma rows must exist).  Run-time compiled only.
        const int act_shape = same_act ? ch.activation : (any_swish ? (int)EH_ACT_SWISH : ch.activation);
        const Variant* vp = (want_jit || !same_act) ? find_shape(Pt, NHmax, rup4(hmax), Ot, act_shape)
                                                    : find_variant(EH_PM_PROGRAM, Pt, NHmax, rup4(hmax), Ot, ch.activation, 1, 0);
        // a shape without a compiled-in variant is compiled at run time without being asked (unless EH_JIT=0): the
        // alternative would be the bf16 path or a refusal
        if (!same_act) {
            auto_jit = !want_jit && !env_jit && vp != nullptr;
            if (!want_jit && !auto_jit) vp = nullptr;
        } else if (!vp && !want_jit && !env_jit) {
            vp = find_shape(Pt, NHmax, rup4(hmax), Ot, ch.activation);
            auto_jit = vp != nullptr;
        }
        if (vp && !same_act) {
            for (int l = 0; l < 3; l++)
                for (int j = 0; j < 32; j++) unit_act[l][j] = (unsigned char)act_shape;
            for (int l = 0; l < NHmax; l++) {
                int u = 0;
                for (int k = 0; k < NC; k++) {
                    const eh_chain_desc& ck = d->chains[k];
                    const int wk = ck.hidden[std::min(l, ck.n_hidden - 1)];
                    for (int j = 0; j < wk && u + j < 32; j++) unit_act[l][u + j] = (unsigned char)(l < ck.n_hidden ? ck.activation : (int)EH_ACT_IDENTITY);
                    u += wk;
                }
            }
        }
        if (vp && vp->NPART <= UPD_MAX_NPART && builtin_as_program(d, is_prog, prog, prog_out)) { v = vp; use_prog = true; }
        if (use_prog) {
            memset(&pd, 0, sizeof pd);
            pd.len = (int)prog.size(); pd.nt = d->n_targ; pd.nf = d->n_forc; pd.np = d->n_params;
            for (int t = 0; t < d->n_targ; t++) pd.out[t] = prog_out[(size_t)t];
            for (int i = 0; i < pd.len; i++) {
                pd.op[i] = (short)prog[(size_t)i].op; pd.a[i] = (short)prog[(size_t)i].a; pd.b[i] = (short)prog[(size_t)i].b;
                pd.imm[i] = prog[(size_t)i].imm;
            }
            if (want_jit || auto_jit) {
                std::string jerr;
                if (jit_compile(pd, *v, same_act ? nullptr : &unit_act[0][0], &c->jit_cubin, c->jit_names, &c->jit.name, &c->jit.from_cache, &c->jit.compile_seconds, &jerr)) {
                    c->jit_on = true;
                } else if (want_jit) {
                    return fail(c, EH_EUNSUPPORTED, "run-time specialisation of the traced process model failed: %s", jerr.c_str());
                } else {
                    v = nullptr; use_prog = false;   // no NVRTC on this machine: the model takes whatever path is left
                }
            }
        }
    }
    // (chains that differ in activation or depth with some layer wider than 32 units: the tensor-core path's per-unit form)
    if (!v && !same_act && hmax <= 32)
        return fail(c, EH_EUNSUPPORTED, "chains that differ in activation need run-time compilation (NVRTC; not with EH_JIT=0) on the exact-fp32 "
                                        "generic kernels: <= 3 hidden layers, summed width <= 32 per layer, <= 12 chain inputs, <= 4 chain outputs");
    if (!v && !same_depth && hmax <= 32)
        return fail(c, EH_EUNSUPPORTED, "chains of different depth run on the exact-fp32 generic kernels only: <= 3 hidden layers, "
                                        "summed width <= 32 per layer, <= 12 chain inputs, <= 4 chain outputs");
    if (!v) return build_plan_wide(c, d, is_prog);
    if (!use_prog && v->T != d->n_targ) return fail(c, EH_EINVAL, "process model yields %d targets, descriptor has %d", v->T, d->n_targ);
    c->var = v;
    c->small_prog = use_prog;
    c->scale_rt = scale_flag;
    if (use_prog) c->h_prog = pd;
    {
        if (c->jit_on) {
            c->jit_var = *v;
            c->jit_var.name = c->jit.name.c_str();
            c->jit_var.prepare = nullptr; c->jit_var.launch_step = nullptr; c->jit_var.launch_eval = nullptr;
            c->jit_var.launch_epoch = nullptr; c->jit_var.epoch_max_grid = nullptr; c->jit_var.epoch_func = nullptr;
            c->jit_on = true;
            c->var = v = &c->jit_var;
        }
    }
    c->var2 = (v->engine == 0 && !c->jit_on) ? find_variant(v->pm, v->P, v->NH, v->H, v->NOUT, v->act, v->scale, 2) : nullptr;
    c->var_tc = (v->engine == 0 && !use_prog && !getenv("EH_NO_TC")) ? find_variant(v->pm, v->P, v->NH, v->H, v->NOUT, v->act, v->scale, 4) : nullptr;
    c->n_pred_raw = d->n_pred; c->n_forc_raw = d->n_forc; c->n_targ = d->n_targ;
    c->use_bn = ch.input_batchnorm ? 1 : 0;
    c->real_in = Pt;
    c->n_chains = NC;
    for (int k = 0, o = 0; k < NC && k < 4; k++) { c->chain_in0[k] = o; c->chain_nin[k] = d->chains[k].n_in; o += d->chains[k].n_in; }
    c->flags = (unsigned)d->flags;

    // flat layout (reference ComponentArray order): chain after chain, per layer W (out x in, column-major) then b; then phi.
    // Level 0 = inputs, 1..NH = hidden layers, L = outputs; chain k owns units [u0[k][lev], u0[k][lev] + cw[k][lev]).
    const ShapeDims& D = v->dims;
    const int L = NHmax + 1;
    std::vector<std::vector<int>> cw((size_t)NC, std::vector<int>((size_t)L + 1)), u0((size_t)NC, std::vector<int>((size_t)L + 1)),
        w_off((size_t)NC, std::vector<int>((size_t)L)), b_off((size_t)NC, std::vector<int>((size_t)L));
    std::vector<int> width((size_t)L + 1, 0);   // embedded (summed) width per level
    int off = 0;
    for (int k = 0; k < NC; k++) {
        const eh_chain_desc& ck = d->chains[k];
        cw[k][0] = ck.n_in;
        for (int l = 0; l < NHmax; l++) cw[k][l + 1] = ck.hidden[std::min(l, ck.n_hidden - 1)];
        cw[k][L] = ck.n_out;
        for (int lev = 0; lev <= L; lev++) { u0[k][lev] = width[lev]; width[lev] += cw[k][lev]; }
        for (int l = 0; l < L; l++) {
            // embedded layers [n_hidden, L-1) of a shallower chain are pass-through: no flat entries (offset -1)
            const bool pass = l >= ck.n_hidden && l < L - 1;
            if (pass) {
                w_off[k][l] = b_off[k][l] = -1;
                for (int j = 0; j < cw[k][l + 1]; j++) c->pass_mask[l] |= 1u << (u0[k][l + 1] + j);
                continue;
            }
            w_off[k][l] = off; off += cw[k][l] * cw[k][l + 1];
            b_off[k][l] = off; off += cw[k][l + 1];
        }
    }
    c->ntheta = off;
    int ng = 0;
    for (int p = 0; p < d->n_params; p++)
        if (d->role[p] == EH_ROLE_GLOBAL) ng = std::max(ng, d->role_index[p] + 1);
    c->nglob = ng;
    c->nflat = off + ng;
    if (!wide && c->nflat > 2048 - NSTAT) return fail(c, EH_EUNSUPPORTED, "parameter vector too long for the single-CTA update");
    // native extra loss lambda * weight_l2(ps.<chains>; normalize) (ABI version 2; extract_weights.jl:55-91,
    // compute_loss.jl:31-34): per flat entry the coefficient of its own value in the gradient, 2 lambda [/ n] for the
    // `weight` entries of the selected chains, 0 elsewhere
    c->l2_on = d->abi_version >= 2 && d->l2_lambda != 0.f;
    if (c->l2_on) {
        long long nw = 0;
        for (int k = 0; k < NC; k++)
            if (!d->l2_chain_mask || ((d->l2_chain_mask >> k) & 1u))
                for (int l = 0; l < L; l++) nw += w_off[k][l] < 0 ? 0 : (long long)cw[k][l] * cw[k][l + 1];
        const double lam = (double)d->l2_lambda / ((d->l2_normalize && nw > 0) ? (double)nw : 1.0);
        c->l2_aggw = d->agg == EH_AGG_MEAN ? 0.5f : 1.0f;
        c->l2_loss_coef = (float)lam;
        c->h_l2coef.assign((size_t)c->nflat, 0.f);
        for (int k = 0; k < NC; k++)
            if (!d->l2_chain_mask || ((d->l2_chain_mask >> k) & 1u))
                for (int l = 0; l < L; l++)
                    for (int i = 0; w_off[k][l] >= 0 && i < cw[k][l] * cw[k][l + 1]; i++) c->h_l2coef[(size_t)w_off[k][l] + i] = (float)(2.0 * lam);
    }

    // smem weight image gather table
    const int H = wide ? v->H : D.H, P = wide ? v->P : D.P, NH = wide ? v->NH : D.NH, NOUT = wide ? v->NOUT : D.NOUT;
    c->h_wsrc.assign((size_t)v->NW + ng, -1);
    if (!wide) {
    // flat entry behind image cell (layer l, embedded output unit j, embedded input unit k); -1: padding or a cell between
    // units of different chains
    auto Wsrc = [&](int l /*1-based*/, int j, int k) -> int {
        for (int q = 0; q < NC; q++) {
            const int jj = j - u0[q][l], kk = k - u0[q][l - 1];
            if (jj >= 0 && jj < cw[q][l] && kk >= 0 && kk < cw[q][l - 1]) {
                if (w_off[q][l - 1] < 0) return jj == kk ? -2 : -1;   // pass-through layer: identity
                return w_off[q][l - 1] + jj + kk * cw[q][l];
            }
        }
        return -1;
    };
    auto Bsrc = [&](int l, int j) -> int {
        for (int q = 0; q < NC; q++) {
            const int jj = j - u0[q][l];
            if (jj >= 0 && jj < cw[q][l]) return b_off[q][l - 1] < 0 ? -1 : b_off[q][l - 1] + jj;
        }
        return -1;
    };
    for (int k = 0; k < P; k++)
        for (int j = 0; j < H; j++) c->h_wsrc[D.off_w1f() + k * H + j] = Wsrc(1, j, k);
    for (int j = 0; j < H; j++) c->h_wsrc[D.off_b1() + j] = Bsrc(1, j);
    for (int l = 2; l <= NH; l++) {
        for (int k = 0; k < H; k++)
            for (int j = 0; j < H; j++) {
                c->h_wsrc[D.off_wf(l) + k * H + j] = Wsrc(l, j, k);
                c->h_wsrc[D.off_wb(l) + j * H + k] = Wsrc(l, j, k);
            }
        for (int j = 0; j < H; j++) c->h_wsrc[D.off_b(l) + j] = Bsrc(l, j);
    }
    for (int o = 0; o < NOUT; o++)
        for (int k = 0; k < H; k++) c->h_wsrc[D.off_wo() + o * H + k] = Wsrc(L, o, k);
    for (int o = 0; o < 4; o++) c->h_wsrc[D.off_bo() + o] = o < NOUT ? Bsrc(L, o) : -1;
    }
    for (int g = 0; g < ng; g++) c->h_wsrc[(size_t)v->NW + g] = off + g;

    // canonical slots from the built-in form's (param, param, forcing) binding
    c->nparam_desc = d->n_params;
    c->slot_of_param.assign((size_t)d->n_params, -1);
    memset(c->slots, 0, sizeof c->slots);
    for (int s = 0; s < MAXPS; s++) c->slots[s].role = ROLE_FIXED;
    for (int s = 0; s < v->NPS; s++) {
        int pi = use_prog ? s : d->pm_args[s].index;   // programs address the parameter table directly
        if (use_prog && pi >= d->n_params) continue;   // unused slot of the generic variant: FIXED, never read
        if (pi < 0 || pi >= d->n_params) return fail(c, EH_EINVAL, "pm_args[%d].index out of range", s);
        PSlot& sl = c->slots[s];
        sl.role = d->role[pi];
        sl.lo = d->lower[pi];
        sl.span = d->upper[pi] - d->lower[pi];
        sl.fixedv = d->deflt[pi];
        if (sl.role == EH_ROLE_NEURAL) {
            const int chain = d->role_index[pi] >> 16, row = d->role_index[pi] & 0xffff;
            if (chain < 0 || chain >= NC || row >= d->chains[chain].n_out)
                return fail(c, EH_EINVAL, "neural parameter %d refers to chain %d row %d", pi, chain, row);
            sl.idx = u0[chain][L] + row;
            if (sl.idx >= NOUT) return fail(c, EH_EINVAL, "neural parameter row %d >= n_out %d", sl.idx, NOUT);
        } else if (sl.role == EH_ROLE_GLOBAL) {
            sl.idx = d->role_index[pi];
        }
        c->slot_of_param[pi] = s;
    }
    for (int i = 0; i < 4; i++) c->pmc[i] = d->pm_consts[i];

    // flat entry -> position in the partial vector
    c->h_pmap.assign((size_t)c->nflat, 0);
    c->h_pspan.assign((size_t)c->nflat, 0.f);
    if (v->engine == 1) {
        // padded-flat partial layout of the tensor-pipe engine (eh_engine_mma.cuh: O_W1 .. O_BO)
        const int o_w1 = 0, o_b1 = H * P, o_w2 = o_b1 + H, o_b2 = o_w2 + H * H, o_wo = o_b2 + H, o_bo = o_wo + NOUT * H;
        const int ow[3] = {o_w1, o_w2, o_wo}, ob[3] = {o_b1, o_b2, o_bo};
        for (int l = 1; l <= L; l++)   // (specialised variants: one chain)
            for (int j = 0; j < width[l]; j++) {
                for (int k = 0; k < width[l - 1]; k++)
                    c->h_pmap[w_off[0][l - 1] + j + k * width[l]] = (l == L) ? ow[2] + j * H + k : ow[l - 1] + j + k * H;
                c->h_pmap[b_off[0][l - 1] + j] = ob[l - 1] + j;
            }
    }
    for (int l = 1; l <= L && v->engine == 0 && !wide; l++) {
        // (jj, kk): unit indices inside chain q; (j, k): the embedded units they live in
        if (l == L && D.LR) {
            // output layer kept in registers: [NOUT][H+1] block behind the statistics
            for (int q = 0; q < NC; q++)
                for (int jj = 0; jj < cw[q][l]; jj++) {
                    const int j = u0[q][l] + jj;
                    for (int kk = 0; kk < cw[q][l - 1]; kk++)
                        c->h_pmap[w_off[q][l - 1] + jj + kk * cw[q][l]] = D.off_last() + j * (H + 1) + u0[q][l - 1] + kk;
                    c->h_pmap[b_off[q][l - 1] + jj] = D.off_last() + j * (H + 1) + H;
                }
            continue;
        }
        const int nk = D.nk(l), b0 = D.blk0(l);
        for (int q = 0; q < NC; q++)
            for (int jj = 0; w_off[q][l - 1] >= 0 && jj < cw[q][l]; jj++) {
                const int j = u0[q][l] + jj;
                for (int kk = 0; kk < cw[q][l - 1]; kk++) {
                    const int k = u0[q][l - 1] + kk;
                    c->h_pmap[w_off[q][l - 1] + jj + kk * cw[q][l]] = (b0 + (j / 4) * nk + (k / 4)) * 16 + (j % 4) * 4 + (k % 4);
                }
                int kb = D.din(l);  // the "ones" row of the augmented input
                c->h_pmap[b_off[q][l - 1] + jj] = (b0 + (j / 4) * nk + (kb / 4)) * 16 + (j % 4) * 4 + (kb % 4);
            }
    }
    for (int g = 0; g < ng; g++) {
        int slot = MAXPS - 1;  // a statistics cell that stays zero (phi not used by the process model)
        float span = 0.f;
        for (int s = 0; s < v->NPS; s++)
            if (c->slots[s].role == ROLE_GLOBAL && c->slots[s].idx == g) { slot = s; span = c->slots[s].span; }
        c->h_pmap[off + g] = v->off_stats + MAXT + slot;
        c->h_pspan[off + g] = span;
    }

    // tables for the persistent kernel: flat parameter -> image cells, phi entry -> slot
    c->h_cells.assign((size_t)2 * c->nflat, -1);
    for (int i = 0; i < v->NW; i++) {
        int p = c->h_wsrc[i];
        if (p < 0) continue;
        if (c->h_cells[2 * p] < 0) c->h_cells[2 * p] = i;
        else c->h_cells[2 * p + 1] = i;
    }
    c->h_slot_of_flat.assign((size_t)c->nflat, -1);
    c->persist_ok = !wide;
    for (int g = 0; g < ng; g++)
        for (int s = 0; s < v->NPS; s++)
            if (c->slots[s].role == ROLE_GLOBAL && c->slots[s].idx == g) c->h_slot_of_flat[off + g] = s;
    c->pm_id = use_prog ? (int)EH_PM_PROGRAM : d->process_model;

    // record columns: chain inputs, the form's forcing, targets.  The generic variants have compile-time maxima:
    // missing inputs / forcings are zero columns (kind 2), missing targets NaN columns (kind 3: always masked)
    c->ncols = 0;
    for (int q = 0; q < NC; q++)
        for (int k = 0; k < d->chains[q].n_in; k++) {
            const int col = d->chains[q].in_cols[k];
            if (col < 0 || col >= d->n_pred) return fail(c, EH_EINVAL, "chain %d in_cols[%d] out of range", q, k);
            c->src_kind[c->ncols] = 0; c->src_idx[c->ncols] = col; c->ncols++;
        }
    for (int k = Pt; k < v->P; k++) { c->src_kind[c->ncols] = 2; c->src_idx[c->ncols] = 0; c->ncols++; }
    if (use_prog) {
        for (int fi = 0; fi < v->F; fi++) {
            c->src_kind[c->ncols] = fi < d->n_forc ? 1 : 2; c->src_idx[c->ncols] = fi < d->n_forc ? fi : 0; c->ncols++;
        }
    } else if (is_prog) {
        for (int fi = 0; fi < d->n_forc; fi++) { c->src_kind[c->ncols] = 1; c->src_idx[c->ncols] = fi; c->ncols++; }
    } else {
        int fi = d->pm_args[2].index;
        if (fi < 0 || fi >= d->n_forc) return fail(c, EH_EINVAL, "forcing index out of range");
        c->src_kind[c->ncols] = 1; c->src_idx[c->ncols] = fi; c->ncols++;
    }
    for (int t = 0; t < d->n_targ; t++) { c->src_kind[c->ncols] = 1; c->src_idx[c->ncols] = d->n_forc + t; c->ncols++; }
    for (int t = d->n_targ; t < v->T; t++) { c->src_kind[c->ncols] = 3; c->src_idx[c->ncols] = 0; c->ncols++; }

    // loss / optimiser.  rmse over several targets and pearsonLoss / kgeLoss / pbkgeLoss need statistics of the batch's
    // predictions before the seeds exist: those targets run as LOSS_AFFINE behind a forward pre-pass (enqueue_stat_prepass)
    for (int t = 0; t < d->n_targ; t++) {
        int lk = d->loss_per_target[t];
        if (lk < 0 || lk > EH_LOSS_PBKGELOSS) return fail(c, EH_EINVAL, "loss_per_target[%d]=%d unknown", t, lk);
        c->loss_kind_abi[t] = lk;
        const bool stat = lk >= EH_LOSS_PEARSONLOSS || (lk == EH_LOSS_RMSE && d->n_targ > 1);
        c->loss_kind[t] = stat ? (int)LOSS_AFFINE : lk;
        c->stat_loss |= stat;
    }
    if (c->l2_on) c->persist_ok = false;   // the extra term lives in k_update
    if (c->stat_loss) {
        if (v->engine != 0)
            return fail(c, EH_EUNSUPPORTED, "rmse over several targets / pearsonLoss / kgeLoss / pbkgeLoss run on the FFMA2 engine (drop EH_FLAG_TENSOR_PIPE)");
        c->persist_ok = false;   // one launch pair (+ pre-pass) per step
    }

    c->agg_mean = d->agg == EH_AGG_MEAN;
    c->opt_kind = d->opt_kind;
    if (c->opt_kind < 0 || c->opt_kind > 3) return fail(c, EH_EINVAL, "opt_kind=%d unknown", d->opt_kind);
    c->adamw_coupled = d->adamw_decay_coupled_eta;
    c->eta = d->eta; c->beta1 = d->beta1; c->beta2 = d->beta2; c->eps = d->eps; c->lambda = d->lambda;
    c->bn_mean.assign((size_t)std::max(Pt, v->P), 0.f);   // padded inputs: statistics of a zero column, never read back
    c->bn_var.assign((size_t)std::max(Pt, v->P), 1.f);
    return EH_OK;
}

}  // namespace rt
}  // namespace eh
