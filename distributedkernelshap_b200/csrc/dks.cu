// libdks.so -- host side of the C ABI declared in include/dks.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC (see build.py)
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "dks_kernels.cuh"
#include "dks_tc.cuh"
#include "dks_shared.cuh"
#include "dks_fused.cuh"
#include "dks_l1.cuh"
#include "dks_wide.cuh"
#include "dks_sampler.cuh"
#include "dks_mlp.cuh"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess)                                                                      \
            return fail(DKS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

#define REQUIRE(cond, ...)                                  \
    do {                                                    \
        if (!(cond)) return fail(DKS_ERR_INVALID, __VA_ARGS__); \
    } while (0)

template <typename T>
int dev_alloc(T** p, size_t count) {
    if (*p) { cudaFree(*p); *p = nullptr; }
    if (count == 0) count = 1;
    CUDA_TRY(cudaMalloc((void**)p, count * sizeof(T)));
    return DKS_OK;
}

template <typename T>
void dev_free(T** p) {
    if (*p) { cudaFree(*p); *p = nullptr; }
}

inline int cdiv(long long a, int b) { return (int)((a + b - 1) / b); }

// frees the device buffers the plan of one M owns (all M when M < 0); the caller has synchronised the stream
void free_plan_allocs(dks_ctx* ctx, int M) {
    for (int m = 0; m <= DKS_MAX_GROUPS; ++m) {
        if (M >= 0 && m != M) continue;
        for (void* q : ctx->plan_allocs[m]) cudaFree(q);
        ctx->plan_allocs[m].clear();
    }
}
bool any_plan_allocs(const dks_ctx* ctx) {
    for (int m = 0; m <= DKS_MAX_GROUPS; ++m) if (!ctx->plan_allocs[m].empty()) return true;
    return false;
}

int bind(dks_ctx* ctx) {
    if (!ctx) return fail(DKS_ERR_INVALID, "null ctx");
    CUDA_TRY(cudaSetDevice(ctx->device));
    return DKS_OK;
}

#define BIND(ctx)                      \
    do {                               \
        int _rc = bind(ctx);           \
        if (_rc != DKS_OK) return _rc; \
    } while (0)

#define TRY(expr)                      \
    do {                               \
        int _rc = (expr);              \
        if (_rc != DKS_OK) return _rc; \
    } while (0)

int ensure_workspace(dks_ctx* ctx, int n) {
    if (n <= ctx->cap_n) return DKS_OK;
    const int G = ctx->G, R = ctx->R, C = ctx->C;
    TRY(dev_alloc(&ctx->d_XW, (size_t)n * G * (ctx->mlp ? ctx->H : R)));
    TRY(dev_alloc(&ctx->d_XT, (size_t)n * ((G + 3) / 4) * 16));
    TRY(dev_alloc(&ctx->d_vflag, (size_t)n * G));
    TRY(dev_alloc(&ctx->d_vmask, (size_t)n));
    TRY(dev_alloc(&ctx->d_M, (size_t)n));
    TRY(dev_alloc(&ctx->d_dlink, (size_t)n * C));
    TRY(dev_alloc(&ctx->d_idx_full, (size_t)n));
    TRY(dev_alloc(&ctx->d_idx_other, (size_t)n));
    TRY(dev_alloc(&ctx->d_acc, (size_t)n * 16));
    TRY(dev_alloc(&ctx->d_done, (size_t)n));
    CUDA_TRY(cudaMemsetAsync(ctx->d_acc, 0, sizeof(long long) * (size_t)n * 16, ctx->stream));   // the fused kernel leaves
    CUDA_TRY(cudaMemsetAsync(ctx->d_done, 0, sizeof(int) * (size_t)n, ctx->stream));             // both zeroed behind it
    ctx->cap_n = n;
    ctx->epoch++;            // buffers moved: a captured graph holds the old addresses
    return DKS_OK;
}

// timing events: inside a stream capture they become external event-record nodes, so dks_last_timings keeps working
// for graph launches
cudaError_t record_ev(dks_ctx* ctx, int k) {
    if (ctx->capturing && !ctx->opt_graph_timing) {   // four event-record nodes cost a replayed graph several microseconds
        ctx->timing_valid = false;
        return cudaSuccess;
    }
    if (k == 0) ctx->timing_valid = true;
    return cudaEventRecordWithFlags(ctx->ev[k], ctx->stream, ctx->capturing ? cudaEventRecordExternal : cudaEventRecordDefault);
}

int launch_prepare(dks_ctx* ctx, const double* X_dev, int n) {
    const int G = ctx->G;
    TRY(ensure_workspace(ctx, n));
    // status word, list counters and the histogram of M are adjacent: one memset
    CUDA_TRY(cudaMemsetAsync(ctx->d_status, 0, sizeof(int) * (4 + G + 1), ctx->stream));
    if (!ctx->capturing) ctx->last_was_graph = false;
    CUDA_TRY(record_ev(ctx, 0));
    if (ctx->mlp) {
        dks::mlp::mlp_prep_kernel<<<n, 128, 0, ctx->stream>>>(
            X_dev, ctx->d_W, ctx->d_b, ctx->d_W2, ctx->d_b2, ctx->d_bg, ctx->d_goff, ctx->d_gcols, ctx->d_colmin,
            ctx->d_colmax, ctx->d_colnan, ctx->d_linkfnull, n, ctx->N, ctx->D, G, ctx->H, ctx->R, ctx->C, ctx->act, ctx->kappa,
            ctx->link, ctx->d_XW, ctx->d_vmask, ctx->d_M, ctx->d_dlink, ctx->d_hist, ctx->d_counts, ctx->d_idx_full,
            ctx->d_idx_other);
        ctx->launches += 1;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(record_ev(ctx, 1));
        ctx->cur_n = n;
        ctx->cur_X = X_dev;
        ctx->prepared = true;
        return DKS_OK;
    }
    int ipb = 256 / G;
    if (ipb < 1) ipb = 1;
    const bool stage = dks::prep_smem_bytes(true, ipb, G, ctx->R, ctx->D) <= (size_t)96 * 1024;
    const size_t psm = dks::prep_smem_bytes(stage, ipb, G, ctx->R, ctx->D);
    auto kern = stage ? dks::prep_kernel<true> : dks::prep_kernel<false>;
    if (psm > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
    kern<<<cdiv(n, ipb), 256, psm, ctx->stream>>>(
        X_dev, ctx->d_W, ctx->d_b, ctx->d_bg, ctx->d_goff, ctx->d_gcols, ctx->d_colmin, ctx->d_colmax, ctx->d_colnan,
        ctx->d_linkfnull, n, ctx->N, ctx->D, G, ctx->R, ctx->C, ctx->act, ctx->kappa, ctx->link, ipb, ctx->d_XW,
        ctx->d_vmask, ctx->d_M, ctx->d_dlink, ctx->d_hist, ctx->d_counts, ctx->d_idx_full, ctx->d_idx_other,
        (ctx->act == DKS_ACT_BINARY_LOGISTIC && ctx->R == 1) ? ctx->d_XT : nullptr, ctx->scale);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(record_ev(ctx, 1));
    ctx->cur_n = n;
    ctx->cur_X = X_dev;
    ctx->prepared = true;
    return DKS_OK;
}

// the solve behind the shared-plan coalition kernels: from the (sum p1, sum p0) buffer of the instances whose groups all
// vary to phi (projection solve, normal-matrix solve, l1 selection, or the float64 product beyond 128 groups)
int launch_sums_solve(dks_ctx* ctx, const PlanDev& pg, int n, double* phi_dev, bool l1) {
    const int G = ctx->G, S = pg.S, S_pad = pg.S_pad;
    dks::shared_path::WlsSharedParams wp;
    wp.n = n; wp.N = ctx->N; wp.G = G; wp.C = ctx->C; wp.S = S; wp.S_pad = S_pad; wp.link = ctx->link;
    wp.uniform_w = 1; wp.sums = ctx->d_sums; wp.z = pg.z; wp.w = pg.w; wp.ainv = pg.ainv; wp.dlink = ctx->d_dlink;
    wp.linkfnull = ctx->d_linkfnull; wp.fnull = ctx->d_fnull; wp.list = ctx->d_idx_full; wp.count = ctx->d_counts;
    wp.phi = phi_dev;
    if (l1) {
        // upstream's l1 branch: moments of y per instance, then the LARS path + criterion + restricted WLS, one warp each
        const dks_ctx::L1Dev& lt = ctx->h_l1[G];
        const size_t need_m = (size_t)n * (2 * G + 4);
        if (need_m > ctx->cap_mom) { TRY(dev_alloc(&ctx->d_mom, need_m)); ctx->cap_mom = need_m; ctx->epoch++; }
        dks::l1::Params lp;
        memset(&lp, 0, sizeof(lp));
        lp.n = n; lp.N = ctx->N; lp.G = G; lp.C = ctx->C; lp.S = S; lp.S_pad = S_pad; lp.link = ctx->link;
        lp.mode = ctx->l1_mode; lp.kfeat = ctx->l1_k; lp.sums = ctx->d_sums; lp.z = pg.z; lp.w = pg.w;
        lp.t.gram_raw = lt.gram_raw; lp.t.gram_norm = lt.gram_norm; lp.t.colsum = lt.colsum; lp.t.scale = lt.scale;
        lp.t.bz = lt.bz; lp.t.gram_w = lt.gram_w; lp.t.b = lt.b; lp.t.sqab = lt.sqab; lp.t.sum_b = lt.sum_b;
        lp.t.sum_sqb = lt.sum_sqb; lp.t.n_aug = lt.n_aug;
        lp.dlink = ctx->d_dlink; lp.linkfnull = ctx->d_linkfnull; lp.fnull = ctx->d_fnull; lp.list = ctx->d_idx_full;
        lp.count = ctx->d_counts; lp.mom = ctx->d_mom; lp.phi = phi_dev; lp.status = ctx->d_status;
        const size_t msm = sizeof(double) * (size_t)S;
        if (msm + 8192 > (size_t)ctx->max_smem_optin)
            return fail(DKS_ERR_UNSUPPORTED, "l1 feature selection: %d coalitions per plan exceed the shared-memory staging", S);
        const int mgrid = n < ctx->sm_count * 2 ? n : ctx->sm_count * 2;
        if (pg.W == 1) {
            CUDA_TRY(cudaFuncSetAttribute(dks::l1::l1_moments_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msm));
            dks::l1::l1_moments_kernel<1><<<mgrid, dks::l1::MOM_THREADS, msm, ctx->stream>>>(lp);
        } else {
            CUDA_TRY(cudaFuncSetAttribute(dks::l1::l1_moments_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msm));
            dks::l1::l1_moments_kernel<2><<<mgrid, dks::l1::MOM_THREADS, msm, ctx->stream>>>(lp);
        }
        const size_t per_warp = dks::l1::lars_smem_per_warp(G);
        const size_t gram_bytes = sizeof(double) * (size_t)G * G;
        const size_t budget = (size_t)ctx->max_smem_optin - 2048;
        // the Gram matrix of the path goes to shared memory when at least four warps still fit next to it
        const int stage_gram = (gram_bytes + 4 * per_warp <= budget) ? 1 : 0;
        int wpc = (int)((budget - (stage_gram ? gram_bytes : 0)) / per_warp);
        if (wpc < 1) return fail(DKS_ERR_UNSUPPORTED, "l1 feature selection: the %d x %d Cholesky factor does not fit shared memory", G, G);
        if (wpc > 8) wpc = 8;
        const size_t lsm = per_warp * wpc + (stage_gram ? gram_bytes : 0);
        int per_sm = (int)((size_t)ctx->max_smem_optin / (lsm + 1024));
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 4) per_sm = 4;
        int lgrid = (n + wpc - 1) / wpc;
        if (lgrid > ctx->sm_count * per_sm) lgrid = ctx->sm_count * per_sm;
        CUDA_TRY(cudaFuncSetAttribute(dks::l1::l1_lars_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm));
        dks::l1::l1_lars_kernel<<<lgrid, 32 * wpc, lsm, ctx->stream>>>(lp, wpc, stage_gram);
    } else if (pg.W > 2) {
        // more than 128 groups: link, float64 product with the host-supplied projection, remainder (dks_wide.cuh)
        const size_t need_y = (size_t)n * S_pad, need_b = (size_t)n * pg.kpw;
        if (need_y > ctx->cap_yw) { TRY(dev_alloc(&ctx->d_yw, need_y)); ctx->cap_yw = need_y; ctx->epoch++; }
        if (need_b > ctx->cap_betaw) { TRY(dev_alloc(&ctx->d_betaw, need_b)); ctx->cap_betaw = need_b; ctx->epoch++; }
        dks::wide::WideParams qp;
        memset(&qp, 0, sizeof(qp));
        qp.n = n; qp.N = ctx->N; qp.G = G; qp.C = ctx->C; qp.S = S; qp.S_pad = S_pad; qp.KP = pg.kpw; qp.link = ctx->link;
        qp.sums = ctx->d_sums; qp.PT = pg.ptw; qp.dvec = pg.dvecw; qp.dlink = ctx->d_dlink;
        qp.linkfnull = ctx->d_linkfnull; qp.fnull = ctx->d_fnull; qp.list = ctx->d_idx_full; qp.count = ctx->d_counts;
        qp.y = ctx->d_yw; qp.beta = ctx->d_betaw; qp.phi = phi_dev;
        CUDA_TRY(dks::wide::launch_wide_solve(qp, n, ctx->sm_count, ctx->opt_wide_gemm, ctx->stream));
        ctx->launches += 2;                      // three launches; the common tail below counts one of them
    } else if (pg.pmat != nullptr) {
        dks::shared_path::WlsPmatParams pp;
        pp.n = n; pp.N = ctx->N; pp.G = G; pp.C = ctx->C; pp.S = S; pp.S_pad = S_pad; pp.link = ctx->link; pp.uniform_w = 1;
        pp.sums = ctx->d_sums; pp.pmat = pg.pmat; pp.dvec = pg.dvec; pp.dlink = ctx->d_dlink;
        pp.linkfnull = ctx->d_linkfnull; pp.fnull = ctx->d_fnull; pp.list = ctx->d_idx_full; pp.count = ctx->d_counts;
        pp.phi = phi_dev;
        cudaError_t perr = cudaSuccess;
        if (!dks::shared_path::launch_wls_pmat(pp, n, ctx->sm_count, ctx->max_smem_optin, ctx->stream, &perr))
            return fail(DKS_ERR_UNSUPPORTED, "projection solve does not fit shared memory");
        CUDA_TRY(perr);
    } else {
        const size_t wsm = dks::shared_path::wls_shared_smem(G);
        int per_sm = (int)((size_t)ctx->max_smem_optin / (wsm + 24 * 1024));
        if (per_sm > 4) per_sm = 4;
        if (per_sm < 1) per_sm = 1;
        int wgrid = n < ctx->sm_count * per_sm ? n : ctx->sm_count * per_sm;   // persistent CTAs of 8 warps
        if (pg.W == 1) {
            CUDA_TRY(cudaFuncSetAttribute(dks::shared_path::wls_shared_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsm));
            dks::shared_path::wls_shared_kernel<1><<<wgrid, dks::shared_path::WLS_THREADS, wsm, ctx->stream>>>(wp);
        } else {
            CUDA_TRY(cudaFuncSetAttribute(dks::shared_path::wls_shared_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsm));
            dks::shared_path::wls_shared_kernel<2><<<wgrid, dks::shared_path::WLS_THREADS, wsm, ctx->stream>>>(wp);
        }
    }
    return DKS_OK;
}

// Coalition stage of a one-hidden-layer ReLU network (dks_mlp.cuh): the shared-plan MLP kernel for the instances whose
// groups all vary (binary head, uniform background weights, the engine's plans), then the linear engine's solve of its
// (sum p1, sum p0) buffer; the general MLP kernel for everything else.  No linear coalition kernel runs on such a context.
int launch_explain_mlp(dks_ctx* ctx, ExplainParams& p, double* phi_dev, bool ext) {
    const int n = ctx->cur_n, G = ctx->G;
    const int kernel = ctx->kernel_choice;
    if (kernel == DKS_KERNEL_TCGEN05)
        return fail(DKS_ERR_UNSUPPORTED, "the tcgen05 kernel evaluates linear models only (this context holds an MLP)");
    dks::mlp::GenParams gp;
    gp.H = ctx->H; gp.BW1 = ctx->d_BW; gp.base1 = ctx->d_scores; gp.W2 = ctx->d_W2; gp.b2 = ctx->d_b2;
    const PlanDev& pg = ctx->h_plans[G];
    const bool fast = (kernel == DKS_KERNEL_AUTO || kernel == DKS_KERNEL_SHARED) && !ext && ctx->act == DKS_ACT_BINARY_LOGISTIC &&
                      ctx->uniform_w && G >= 2 && pg.mlp_dT != nullptr && pg.S == dks_effective_S(G, ctx->nsamples_req);
    if (kernel == DKS_KERNEL_SHARED && !fast && !ext && pg.z != nullptr)
        return fail(DKS_ERR_UNSUPPORTED, "shared-plan MLP kernel needs the binary-logistic head, uniform background weights, "
                    "at most %d hidden units after sign padding and at most %d background rows", dks::mlp::MAX_H,
                    dks::mlp::FAST_MAXN);
    const bool l1 = ctx->l1_mode != 0;
    if (l1) {
        if (ext || ctx->plan_mode == 1) return fail(DKS_ERR_UNSUPPORTED, "l1 feature selection runs on shared plans only");
        if (!fast || ctx->h_l1[G].gram_raw == nullptr || ctx->h_l1[G].S != pg.S)
            return fail(DKS_ERR_UNSUPPORTED, "l1 feature selection needs the shared-plan path (binary-logistic head, uniform "
                        "background weights) and the l1 tables of the M=%d plan (dks_set_l1_tables)", G);
    }
    cudaStream_t gstream = ctx->stream;
    if (fast && ctx->side_stream != nullptr) {
        CUDA_TRY(cudaEventRecord(ctx->ev_fork, ctx->stream));
        CUDA_TRY(cudaStreamWaitEvent(ctx->side_stream, ctx->ev_fork, 0));
        gstream = ctx->side_stream;
    }
    auto join = [&]() -> cudaError_t {
        if (gstream == ctx->stream) return cudaSuccess;
        cudaError_t e = cudaEventRecord(ctx->ev_join, gstream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0);
        return e;
    };
    if (fast) {
        const int S = pg.S, S_pad = pg.S_pad, HP = ctx->mlp_hp;
        const size_t need = (size_t)n * S_pad;
        if (need > ctx->cap_sums) { TRY(dev_alloc(&ctx->d_sums, need)); ctx->cap_sums = need; ctx->epoch++; }
        // a'(q, s, u) goes through a workspace of at most 1 GiB: chunks of QC instances
        const size_t per_inst = (size_t)S_pad * HP;
        int QC = (int)(((size_t)1 << 28) / per_inst) / 32 * 32;
        if (QC < 32) QC = 32;
        if (QC > (n + 31) / 32 * 32) QC = (n + 31) / 32 * 32;
        const size_t need_a = (size_t)QC * per_inst;
        if (need_a > ctx->cap_mlp_atab) { TRY(dev_alloc(&ctx->d_mlp_atab, need_a)); ctx->cap_mlp_atab = need_a; ctx->epoch++; }
        dks::mlp::SharedParams sp;
        memset(&sp, 0, sizeof(sp));
        sp.N = ctx->N; sp.G = G; sp.H = ctx->H; sp.HP = HP; sp.S = S; sp.S_pad = S_pad; sp.QC = QC;
        sp.scale = ctx->scale; sp.b2 = ctx->h_b2[0]; sp.negmask = ctx->mlp_negmask;
        sp.dT = pg.mlp_dT; sp.Ld = pg.mlp_Ld; sp.z = pg.z; sp.XW = ctx->d_XW; sp.perm = ctx->d_mlp_perm;
        sp.w2abs = ctx->d_mlp_w2abs; sp.atab = ctx->d_mlp_atab; sp.list = ctx->d_idx_full; sp.count = ctx->d_counts;
        sp.sums = ctx->d_sums;
        const size_t asm_bytes = sizeof(float) * (size_t)G * HP;
        const size_t ssm = dks::mlp::shared_smem_bytes(ctx->N, HP);
        CUDA_TRY(cudaFuncSetAttribute(dks::mlp::mlp_atab_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)asm_bytes));
        auto skern = dks::mlp::mlp_shared_kernel<16>;
        switch (HP) {
            case 16: skern = dks::mlp::mlp_shared_kernel<16>; break;
            case 32: skern = dks::mlp::mlp_shared_kernel<32>; break;
            case 48: skern = dks::mlp::mlp_shared_kernel<48>; break;
            case 64: skern = dks::mlp::mlp_shared_kernel<64>; break;
            case 80: skern = dks::mlp::mlp_shared_kernel<80>; break;
            case 96: skern = dks::mlp::mlp_shared_kernel<96>; break;
            case 112: skern = dks::mlp::mlp_shared_kernel<112>; break;
            case 128: skern = dks::mlp::mlp_shared_kernel<128>; break;
            default: return fail(DKS_ERR_INVALID, "MLP unit order of %d units", HP);
        }
        CUDA_TRY(cudaFuncSetAttribute(skern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssm));
        for (int q0 = 0; q0 < n; q0 += QC) {
            sp.q0 = q0;
            dks::mlp::mlp_atab_kernel<<<QC, 256, asm_bytes, ctx->stream>>>(sp);
            skern<<<S, 128, ssm, ctx->stream>>>(sp);
            ctx->launches += 2;
        }
        CUDA_TRY(cudaGetLastError());
        TRY(launch_sums_solve(ctx, pg, n, phi_dev, l1));
        ctx->launches += 1;
        CUDA_TRY(cudaGetLastError());
        p.list = ctx->d_idx_other;      // the general kernel below takes the remaining instances
        p.count = ctx->d_counts + 1;
    }
    if (l1 && !ctx->l1_others_plain) {
        // instances with a partial varying set would need their own selection: reported, not computed
        dks::flag_unsupported_kernel<<<1, 1, 0, gstream>>>(ctx->d_counts + 1, G, ctx->d_status);
    } else {
        const int nacc = dks::mlp::gen_nacc(ctx->act, ctx->C);
        const size_t smem = dks::mlp::gen_smem_bytes(p.S_cap, G < 64 ? G : 64, ctx->R, nacc);
        if ((long long)smem > (long long)ctx->max_smem_optin)
            return fail(DKS_ERR_UNSUPPORTED, "general MLP kernel needs %zu B of shared memory (> %d): nsamples too large", smem,
                        ctx->max_smem_optin);
        CUDA_TRY(cudaFuncSetAttribute(dks::mlp::mlp_general_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = (int)((size_t)ctx->max_smem_optin / (smem + 1024));
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 8) per_sm = 8;
        int grid = ctx->sm_count * per_sm;
        if (grid > n) grid = n;
        dks::mlp::mlp_general_kernel<<<grid, dks::mlp::GEN_THREADS, smem, gstream>>>(p, gp);
    }
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(join());
    return DKS_OK;
}

int launch_explain(dks_ctx* ctx, double* phi_dev, const uint64_t* ext_z, const double* ext_w, int ext_stride) {
    REQUIRE(ctx->prepared, "dks_explain: call dks_prepare_* first");
    REQUIRE((ext_z == nullptr) == (ext_w == nullptr), "ext_zbits and ext_w must both be given or both be NULL");
    const int n = ctx->cur_n;
    const double* ext_chol = nullptr;
    const double* ext_ainv = nullptr;
    int ext_fstride = 0;
    if (ctx->G > 64 && (ext_z != nullptr || ctx->plan_mode == 1))
        return fail(DKS_ERR_UNSUPPORTED, "more than 64 groups: only shared plans are supported (no per-instance plans)");
    if (ctx->plan_mode == 1 && ext_z == nullptr) {
        // every instance draws its own plan on the device; the explain kernels then read it like a caller-supplied one
        if (ctx->max_plan_S < 2)
            return fail(DKS_ERR_PLAN_MISSING, "per-instance plans need the shared plans of the M values present (their "
                        "enumerated prefix); none is set");
        const int stride = (ctx->max_plan_S + 1) & ~1;
        const size_t need = (size_t)n * stride;
        if (need > ctx->cap_gen) {
            TRY(dev_alloc(&ctx->d_genz, need)); TRY(dev_alloc(&ctx->d_genw, need));
            ctx->cap_gen = need; ctx->epoch++;
        }
        const int nAmax = ctx->G > 1 ? ctx->G - 1 : 1;
        const int fstride = nAmax * nAmax;
        const size_t needf = (size_t)n * fstride;
        if (needf > ctx->cap_genf) {
            TRY(dev_alloc(&ctx->d_genchol, needf)); TRY(dev_alloc(&ctx->d_genainv, needf));
            ctx->cap_genf = needf; ctx->epoch++;
        }
        REQUIRE(ctx->d_sinfo && ctx->d_afix, "per-instance plans: dks_set_plan_sampling has not been called");
        // table sized for the largest sampled part among the plans set (a plan's sampled rows <= its S)
        int max_left = 32;
        for (int M = 2; M <= ctx->G && M <= DKS_MAX_GROUPS; ++M)
            if (ctx->h_plans[M].z && ctx->h_sinfo[M].ncdf > 0) {
                const int left = ctx->h_plans[M].S - ctx->h_sinfo[M].nfixed;
                if (left > max_left) max_left = left;
            }
        max_left = (max_left + 31) / 32 * 32;
        if (max_left > dks::sampler::MAX_SAMPLED)
            return fail(DKS_ERR_UNSUPPORTED, "per-instance plans: %d sampled rows per plan exceed the sampler's limit of %d",
                        max_left, dks::sampler::MAX_SAMPLED);
        int cap = 256;                       // hash slots; its arrays are reused for the bit-transposed plan and pair counts
        while (cap < 2 * max_left || cap < nAmax * (nAmax + 1) / 2) cap <<= 1;
        dks::sampler::SamplerParams sp;
        sp.n = n; sp.G = ctx->G; sp.S_req = ctx->nsamples_req; sp.stride = stride; sp.seed = ctx->sampler_seed;
        sp.table_cap = cap; sp.max_left = max_left; sp.fstride = fstride;
        sp.row_offset = ctx->row_offset; sp.Mcnt = ctx->d_M; sp.plans = ctx->d_plans; sp.info = ctx->d_sinfo;
        sp.afix = ctx->d_afix;
        sp.out_z = ctx->d_genz; sp.out_w = ctx->d_genw; sp.out_chol = ctx->d_genchol; sp.out_ainv = ctx->d_genainv;
        sp.status = ctx->d_status;
        const size_t ssm = dks::sampler::smem_bytes(cap, max_left, ctx->G);
        if (ssm + 2048 > (size_t)ctx->max_smem_optin)
            return fail(DKS_ERR_UNSUPPORTED, "per-instance plan sampler needs %zu B of shared memory", ssm);
        CUDA_TRY(cudaFuncSetAttribute(dks::sampler::sample_plans_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssm));
        int per_sm = (int)((size_t)ctx->max_smem_optin / (ssm + 2048));
        if (per_sm > 6) per_sm = 6;
        if (per_sm < 1) per_sm = 1;
        const int sgrid = n < ctx->sm_count * per_sm ? n : ctx->sm_count * per_sm;
        dks::sampler::sample_plans_kernel<<<sgrid, dks::sampler::THREADS, ssm, ctx->stream>>>(sp);
        {
            const size_t per_warp = (size_t)2 * nAmax * nAmax * sizeof(double);
            int fw = (int)((size_t)ctx->max_smem_optin / per_warp);
            if (fw > dks::sampler::FACTOR_WARPS) fw = dks::sampler::FACTOR_WARPS;
            if (fw < 1)
                return fail(DKS_ERR_UNSUPPORTED, "per-instance plans: normal-matrix workspace does not fit shared memory");
            const size_t fsm = (size_t)fw * per_warp;
            CUDA_TRY(cudaFuncSetAttribute(dks::sampler::factor_plans_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsm));
            int fgrid = (n + fw - 1) / fw;
            dks::sampler::factor_plans_kernel<<<fgrid, fw * 32, fsm, ctx->stream>>>(n, ctx->d_M, fstride, ctx->d_genchol,
                                                                                    ctx->d_genainv, nAmax, ctx->d_status);
        }
        ctx->launches += 2;
        CUDA_TRY(cudaGetLastError());
        ctx->gen_stride = stride; ctx->gen_n = n;
        ext_z = ctx->d_genz; ext_w = ctx->d_genw; ext_stride = stride;
        ext_chol = ctx->d_genchol; ext_ainv = ctx->d_genainv; ext_fstride = fstride;
    }
    ExplainParams p;
    memset(&p, 0, sizeof(p));
    p.n = n; p.N = ctx->N; p.G = ctx->G; p.R = ctx->R; p.C = ctx->C;
    p.act = ctx->act; p.link = ctx->link; p.S_req = ctx->nsamples_req;
    p.scale = ctx->scale;
    p.BWs = ctx->d_BWs; p.bases = ctx->d_bases; p.wbf = ctx->d_wbf; p.wbg = ctx->d_wbg; p.Bbar = ctx->d_Bbar;
    p.fnull = ctx->d_fnull; p.linkfnull = ctx->d_linkfnull;
    p.XW = ctx->d_XW; p.vmask = ctx->d_vmask; p.Mcnt = ctx->d_M; p.dlink = ctx->d_dlink;
    p.plans = ctx->d_plans; p.ext_z = ext_z; p.ext_w = ext_w; p.ext_stride = ext_stride;
    p.ext_chol = ext_chol; p.ext_ainv = ext_ainv; p.ext_fstride = ext_fstride;
    p.phi = phi_dev; p.status = ctx->d_status;
    // capacity of the per-CTA y buffer: the largest S any instance can need
    int S_cap = 0;
    if (ext_z) S_cap = ext_stride;
    else S_cap = ctx->max_plan_S;
    if (S_cap < 2) S_cap = 2;
    p.S_cap = S_cap;

    if (ctx->dbg_i >= 0) {   // debug dump of one instance's accumulator tile (tcgen05 kernel only)
        int rows = S_cap, cols = dks::tc_npad(ctx->N);
        if (rows != ctx->dbg_rows || cols != ctx->dbg_cols) {
            TRY(dev_alloc(&ctx->dbg_T, (size_t)rows * cols));
            ctx->dbg_rows = rows; ctx->dbg_cols = cols;
        }
        CUDA_TRY(cudaMemsetAsync(ctx->dbg_T, 0, sizeof(float) * rows * cols, ctx->stream));
        if (!ctx->dbg_time) TRY(dev_alloc(&ctx->dbg_time, (size_t)6 * 256));
        CUDA_TRY(cudaMemsetAsync(ctx->dbg_time, 0, sizeof(float) * 6 * 256, ctx->stream));
    }

    int kernel = ctx->kernel_choice;
    CUDA_TRY(record_ev(ctx, 2));
    if (ctx->mlp) {
        TRY(launch_explain_mlp(ctx, p, phi_dev, ext_z != nullptr));
        CUDA_TRY(record_ev(ctx, 3));
        return DKS_OK;
    }

    // ---- shared-plan fast path: instances whose varying set is all G groups, evaluated against the plan's Dm table
    const int G = ctx->G;
    const PlanDev& pg = ctx->h_plans[G <= DKS_MAX_GROUPS ? G : 0];
    const bool fast = (kernel == DKS_KERNEL_AUTO || kernel == DKS_KERNEL_SHARED) && ext_z == nullptr &&
                      ctx->act == DKS_ACT_BINARY_LOGISTIC && ctx->uniform_w && G >= 2 && pg.dmT != nullptr &&
                      pg.S == dks_effective_S(G, ctx->nsamples_req) && (pg.W <= 2 || pg.ptw != nullptr);
    if (kernel == DKS_KERNEL_SHARED && !fast && ext_z == nullptr && pg.z != nullptr)
        return fail(DKS_ERR_UNSUPPORTED, "shared-plan fast path needs the binary-logistic head and uniform background weights");
    // the general kernel below (instances that are not on the shared-plan path) forks off here and joins at the end
    cudaStream_t gstream = ctx->stream;
    if (fast && ctx->side_stream != nullptr) {
        CUDA_TRY(cudaEventRecord(ctx->ev_fork, ctx->stream));
        CUDA_TRY(cudaStreamWaitEvent(ctx->side_stream, ctx->ev_fork, 0));
        gstream = ctx->side_stream;
    }
    auto join = [&]() -> cudaError_t {
        if (gstream == ctx->stream) return cudaSuccess;
        cudaError_t e = cudaEventRecord(ctx->ev_join, gstream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0);
        return e;
    };
    dks::shared_path::FusedConfig fcfg;
    const bool l1 = ctx->l1_mode != 0;
    if (l1) {
        if (ext_z != nullptr || ctx->plan_mode == 1)
            return fail(DKS_ERR_UNSUPPORTED, "l1 feature selection runs on shared plans only");
        if (pg.W > 2)
            return fail(DKS_ERR_UNSUPPORTED, "l1 feature selection covers plans of at most 128 groups (M=%d)", G);
        if (!fast || ctx->h_l1[G].gram_raw == nullptr || ctx->h_l1[G].S != pg.S)
            return fail(DKS_ERR_UNSUPPORTED, "l1 feature selection needs the shared-plan path (binary-logistic head, uniform "
                        "background weights) and the l1 tables of the M=%d plan (dks_set_l1_tables)", G);
    }
    const bool fused = fast && !l1 && ctx->opt_fused && pg.pmat64 != nullptr && pg.W == 1 &&
                       dks::shared_path::fused_config(ctx->N, G, pg.S_pad, ctx->sm_count, ctx->max_smem_optin,
                                                      ctx->opt_fused_ni, ctx->opt_fused_warps, ctx->opt_fused_B, &fcfg);
    ctx->last_fused = fused;
    if (fused) {
        // link + projection solve inside the coalition kernel: no (sum p1, sum p0) buffer, no separate solve launch
        dks::shared_path::FusedParams fp;
        memset(&fp, 0, sizeof(fp));
        fp.n = n; fp.N = ctx->N; fp.G = G; fp.C = ctx->C; fp.S = pg.S; fp.S_pad = pg.S_pad; fp.link = ctx->link; fp.B = fcfg.B;
        fp.scale = ctx->scale; fp.DmT = pg.dmT; fp.dme = pg.dme; fp.z = pg.z; fp.XT = ctx->d_XT; fp.list = ctx->d_idx_full;
        fp.count = ctx->d_counts; fp.pmat64 = pg.pmat64; fp.dvec = pg.dvec64; fp.dlink = ctx->d_dlink;
        fp.linkfnull = ctx->d_linkfnull; fp.fnull = ctx->d_fnull; fp.acc = ctx->d_acc; fp.done = ctx->d_done; fp.phi = phi_dev;
        if (ctx->peer_world > 1 && ctx->push_in_kernel) {
            double* slabs[16];
            int np = 0;
            for (int r = 0; r < ctx->peer_world; ++r) {
                double* slab = ctx->peer_base[r] + (long long)ctx->peer_rank * ctx->peer_slab;
                if (slab == phi_dev) continue;               // phi is written in place into the local slab
                slabs[np++] = slab;
            }
            if (!ctx->d_peer_list) TRY(dev_alloc(&ctx->d_peer_list, (size_t)16));
            if (ctx->peer_list_for != phi_dev) {             // (never during a capture: the graph key holds the phi pointer)
                CUDA_TRY(cudaMemcpy(ctx->d_peer_list, slabs, sizeof(double*) * np, cudaMemcpyHostToDevice));
                ctx->peer_list_for = phi_dev;
            }
            fp.npeers = np;
            fp.peer_phi = ctx->d_peer_list;
        }
        CUDA_TRY(dks::shared_path::launch_explain_fused(fp, fcfg, ctx->sm_count, ctx->stream));
        ctx->launches += 1;
        CUDA_TRY(cudaGetLastError());
        p.list = ctx->d_idx_other;
        p.count = ctx->d_counts + 1;
    } else if (fast) {
        const int S = pg.S, S_pad = pg.S_pad;
        size_t need = (size_t)n * S_pad;
        if (need > ctx->cap_sums) { TRY(dev_alloc(&ctx->d_sums, need)); ctx->cap_sums = need; ctx->epoch++; }
        dks::shared_path::SharedParams sp;
        sp.n = n; sp.N = ctx->N; sp.G = G; sp.S = S; sp.S_pad = S_pad; sp.scale = ctx->scale;
        sp.DmT = pg.dmT; sp.dme = pg.dme; sp.z = pg.z; sp.XT = ctx->d_XT; sp.list = ctx->d_idx_full; sp.count = ctx->d_counts; sp.sums = ctx->d_sums; sp.accumulate = 0;
        sp.acache = nullptr; sp.acache_mode = 0;
        if (pg.W > 2 && ctx->opt_wide_acache && ctx->N > dks::shared_path::MAXN) {
            // sixteen-word rows, several background chunks: A(i, s) is computed by the first chunk's launch only
            if (need > ctx->cap_acache) { TRY(dev_alloc(&ctx->d_acache, need)); ctx->cap_acache = need; ctx->epoch++; }
            sp.acache = ctx->d_acache;
        }
        ctx->launches += dks::shared_path::launch_explain_shared(sp, pg.W, ctx->sm_count, ctx->stream) - 1;
        TRY(launch_sums_solve(ctx, pg, n, phi_dev, l1));
        ctx->launches += 2;
        CUDA_TRY(cudaGetLastError());
        p.list = ctx->d_idx_other;      // the general kernel below takes the remaining instances
        p.count = ctx->d_counts + 1;
    }
    if (l1 && !ctx->l1_others_plain) {
        // instances with a partial varying set would need their own selection: reported, not computed
        dks::flag_unsupported_kernel<<<1, 1, 0, gstream>>>(ctx->d_counts + 1, G, ctx->d_status);
        ctx->launches += 1;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(join());
        CUDA_TRY(record_ev(ctx, 3));
        return DKS_OK;
    }
    if (G > 64) {
        // two-word coalition rows exist on the shared-plan path only: anything left over is reported, not computed
        if (pg.z == nullptr || pg.S != dks_effective_S(G, ctx->nsamples_req) || (pg.W > 2 && pg.ptw == nullptr)) {
            ctx->h_status[0] = DKS_ERR_PLAN_MISSING; ctx->h_status[1] = G;
            return fail(DKS_ERR_PLAN_MISSING, "no shared plan for M=%d at the current nsamples", G);
        }
        if (!fast)
            return fail(DKS_ERR_UNSUPPORTED, "more than 64 groups needs the shared-plan path (binary-logistic head, uniform "
                        "background weights, kernel 'auto' or 'shared', shared plan of M=%d uploaded)", G);
        dks::flag_unsupported_kernel<<<1, 1, 0, gstream>>>(ctx->d_counts + 1, G, ctx->d_status);
        ctx->launches += 1;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(join());
        CUDA_TRY(record_ev(ctx, 3));
        return DKS_OK;
    }
    if (kernel == DKS_KERNEL_AUTO || kernel == DKS_KERNEL_SHARED)
        kernel = dks::tc_supported(ctx, p) ? DKS_KERNEL_TCGEN05 : DKS_KERNEL_SIMT;
    if (kernel == DKS_KERNEL_TCGEN05) {
        if (!dks::tc_supported(ctx, p))
            return fail(DKS_ERR_UNSUPPORTED, "tcgen05 kernel does not support this shape/head (N=%d G=%d act=%d)", ctx->N,
                        ctx->G, ctx->act);
        TRY(dks::tc_launch(ctx, p, gstream));
    } else {
        const bool sfm = ctx->act == DKS_ACT_SOFTMAX;
        size_t smem = dks::simt_smem_bytes(S_cap, ctx->N, ctx->G, sfm ? ctx->R : 1, sfm ? ctx->C : 1);
        if ((long long)smem > (long long)ctx->max_smem_optin)
            return fail(DKS_ERR_UNSUPPORTED, "SIMT kernel needs %zu B of shared memory (> %d): N*G or nsamples too large",
                        smem, ctx->max_smem_optin);
        CUDA_TRY(cudaFuncSetAttribute(dks::explain_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = (int)((size_t)ctx->max_smem_optin / (smem + 1024));
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 8) per_sm = 8;
        int grid = ctx->sm_count * per_sm;
        if (grid > n) grid = n;
        dks::explain_simt_kernel<<<grid, 256, smem, gstream>>>(p);
        ctx->launches += 1;
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(join());
    CUDA_TRY(record_ev(ctx, 3));
    return DKS_OK;
}

int check_status(dks_ctx* ctx) {
    // status was copied to h_status by the caller and the stream synchronised
    if (ctx->h_status[0] == 0) return DKS_OK;
    if (ctx->h_status[0] == DKS_ERR_PLAN_MISSING)
        return fail(DKS_ERR_PLAN_MISSING, "no shared plan for M=%d at the current nsamples", ctx->h_status[1]);
    if (ctx->h_status[0] == DKS_ERR_NUMERIC)
        return fail(DKS_ERR_NUMERIC, "normal matrix not positive definite (instance/M %d)", ctx->h_status[1]);
    return fail(ctx->h_status[0], "explain kernel reported status %d (detail %d)", ctx->h_status[0], ctx->h_status[1]);
}

}  // namespace

extern "C" {

int dks_version(void) { return DKS_VERSION; }

const char* dks_last_error(void) { return g_last_error.c_str(); }

int dks_device_count(int* count) {
    if (!count) return fail(DKS_ERR_INVALID, "dks_device_count: NULL");
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); c = 0; }
    *count = c;
    return DKS_OK;
}

int dks_create(dks_ctx** out, int device) {
    if (!out) return fail(DKS_ERR_INVALID, "dks_create: out is NULL");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(DKS_ERR_CUDA, "dks_create: no CUDA device (%s) -- the engine has no CPU fallback",
                    cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(DKS_ERR_INVALID, "dks_create: device %d out of range [0,%d)", device, count);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(DKS_ERR_UNSUPPORTED, "dks_create: device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    dks_ctx* ctx = new dks_ctx();
    ctx->device = device;
    { const char* e = getenv("DKS_GRAPH"); ctx->graph_enabled = !(e && e[0] == '0'); }
    {
        auto env_int = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
        ctx->opt_fused = env_int("DKS_FUSED", 1);
        ctx->opt_fused_ni = env_int("DKS_FUSED_NI", 0);
        ctx->opt_fused_warps = env_int("DKS_FUSED_WARPS", 0);
        ctx->opt_fused_B = env_int("DKS_FUSED_B", 0);
        ctx->push_in_kernel = env_int("DKS_PUSH_IN_KERNEL", 0) != 0;
        ctx->opt_wide_gemm = env_int("DKS_WIDE_GEMM", ctx->opt_wide_gemm) == 2 ? 2 : 1;
        ctx->opt_wide_acache = env_int("DKS_WIDE_ACACHE", ctx->opt_wide_acache ? 1 : 0) != 0;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    memset(ctx->h_plans, 0, sizeof(ctx->h_plans));
    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
    for (int i = 0; i < 4; ++i) CUDA_TRY(cudaEventCreate(&ctx->ev[i]));
    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    CUDA_TRY(cudaMalloc((void**)&ctx->d_plans, sizeof(ctx->h_plans)));
    CUDA_TRY(cudaMemset(ctx->d_plans, 0, sizeof(ctx->h_plans)));
    CUDA_TRY(cudaMalloc((void**)&ctx->d_status, sizeof(int) * (4 + DKS_MAX_GROUPS + 1)));   // status, list counts, histogram
    ctx->d_counts = ctx->d_status + 2;
    ctx->d_hist = ctx->d_status + 4;
    CUDA_TRY(cudaMemset(ctx->d_status, 0, sizeof(int) * (4 + DKS_MAX_GROUPS + 1)));
    *out = ctx;
    return DKS_OK;
}

int dks_destroy(dks_ctx* ctx) {
    if (!ctx) return DKS_OK;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->gexec) { cudaGraphExecDestroy(ctx->gexec); ctx->gexec = nullptr; }
    dev_free(&ctx->d_bg); dev_free(&ctx->d_wbg); dev_free(&ctx->d_W); dev_free(&ctx->d_b);
    dev_free(&ctx->d_goff); dev_free(&ctx->d_gcols); dev_free(&ctx->d_colmin); dev_free(&ctx->d_colmax);
    dev_free(&ctx->d_colnan); dev_free(&ctx->d_BW); dev_free(&ctx->d_scores); dev_free(&ctx->d_Bbar);
    dev_free(&ctx->d_fnull); dev_free(&ctx->d_linkfnull); dev_free(&ctx->d_BWs); dev_free(&ctx->d_bases);
    dev_free(&ctx->d_wbf); dev_free(&ctx->d_plans); dev_free(&ctx->d_X); dev_free(&ctx->d_XW); dev_free(&ctx->d_XT);
    dev_free(&ctx->d_vflag); dev_free(&ctx->d_vmask); dev_free(&ctx->d_M); dev_free(&ctx->d_dlink);
    dev_free(&ctx->d_idx_full); dev_free(&ctx->d_idx_other); dev_free(&ctx->d_sums); dev_free(&ctx->d_acc); dev_free(&ctx->d_done); dev_free(&ctx->d_mom); dev_free(&ctx->d_step); dev_free(&ctx->d_peer_list);
    dev_free(&ctx->d_status); ctx->d_hist = nullptr; ctx->d_counts = nullptr; dev_free(&ctx->d_yw); dev_free(&ctx->d_betaw); dev_free(&ctx->d_acache); dev_free(&ctx->d_phi); if (ctx->h_phi_pin) { cudaFreeHost(ctx->h_phi_pin); ctx->h_phi_pin = nullptr; } dev_free(&ctx->d_genz); dev_free(&ctx->d_genw); dev_free(&ctx->d_genchol); dev_free(&ctx->d_genainv); dev_free(&ctx->d_afix); dev_free(&ctx->d_sinfo); dev_free(&ctx->d_extz);
    dev_free(&ctx->d_extw);
    dev_free(&ctx->d_W2); dev_free(&ctx->d_b2); dev_free(&ctx->d_mlp_perm); dev_free(&ctx->d_mlp_w2abs);
    dev_free(&ctx->d_mlp_atab);
    dev_free(&ctx->dbg_T);
    dev_free(&ctx->dbg_time);
    free_plan_allocs(ctx, -1);
    for (int i = 0; i < 4; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->side_stream) cudaStreamDestroy(ctx->side_stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return DKS_OK;
}

int dks_set_stream(dks_ctx* ctx, void* stream) {
    BIND(ctx);
    if (ctx->own_stream && ctx->stream) {
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        CUDA_TRY(cudaStreamDestroy(ctx->stream));
    }
    ctx->stream = (cudaStream_t)stream;
    ctx->own_stream = false;
    return DKS_OK;
}

int dks_synchronize(dks_ctx* ctx) {
    BIND(ctx);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DKS_OK;
}

int dks_set_background(dks_ctx* ctx, const double* bg_host, int N, int D, const double* weights_host) {
    BIND(ctx);
    REQUIRE(bg_host && N > 0 && D > 0, "dks_set_background: need bg, N > 0, D > 0");
    ctx->N = N; ctx->D = D;
    ctx->h_bg.assign(bg_host, bg_host + (size_t)N * D);
    ctx->h_wbg.assign(N, 1.0 / N);
    ctx->uniform_w = true;
    if (weights_host) {
        for (int j = 1; j < N; ++j) if (weights_host[j] != weights_host[0]) ctx->uniform_w = false;
        double sum = 0;
        for (int j = 0; j < N; ++j) sum += weights_host[j];
        REQUIRE(sum > 0, "dks_set_background: weights must have a positive sum");
        for (int j = 0; j < N; ++j) ctx->h_wbg[j] = weights_host[j] / sum;
    }
    ctx->fitted = false;
    return DKS_OK;
}

int dks_set_groups(dks_ctx* ctx, const int32_t* group_offsets, const int32_t* group_cols, int G) {
    BIND(ctx);
    REQUIRE(group_offsets && group_cols && G > 0, "dks_set_groups: need offsets, cols, G > 0");
    if (G > DKS_MAX_GROUPS)
        return fail(DKS_ERR_UNSUPPORTED, "dks_set_groups: G=%d groups; this build handles at most %d (sixteen 64-bit words "
                    "of coalition bits per row)", G, DKS_MAX_GROUPS);
    ctx->G = G;
    ctx->h_goff.assign(group_offsets, group_offsets + G + 1);
    ctx->h_gcols.assign(group_cols, group_cols + group_offsets[G]);
    ctx->fitted = false;
    return DKS_OK;
}

int dks_set_model(dks_ctx* ctx, const double* W_host, const double* b_host, int R, int activation, double kappa,
                  int scalar_out) {
    BIND(ctx);
    REQUIRE(ctx->D > 0, "dks_set_model: call dks_set_background first (D unknown)");
    REQUIRE(W_host && b_host && R > 0, "dks_set_model: need W, b, R > 0");
    if (R > 8) return fail(DKS_ERR_UNSUPPORTED, "dks_set_model: R=%d score rows; at most 8 supported", R);
    if (activation == DKS_ACT_BINARY_LOGISTIC) {
        REQUIRE(R == 1, "binary-logistic head needs R == 1 (got %d)", R);
        REQUIRE(kappa > 0, "binary-logistic head needs kappa > 0");
        ctx->C = 2;
    } else if (activation == DKS_ACT_IDENTITY) {
        ctx->C = R;
    } else if (activation == DKS_ACT_SOFTMAX) {
        REQUIRE(R >= 2, "softmax head needs at least two score rows (got %d)", R);
        ctx->C = R;
    } else {
        return fail(DKS_ERR_INVALID, "dks_set_model: unknown activation %d", activation);
    }
    ctx->R = R; ctx->act = activation; ctx->kappa = kappa; ctx->scalar_out = scalar_out;
    ctx->h_W.assign(W_host, W_host + (size_t)R * ctx->D);
    ctx->h_b.assign(b_host, b_host + R);
    ctx->mlp = false;
    ctx->fitted = false;
    return DKS_OK;
}

int dks_set_mlp_model(dks_ctx* ctx, const double* W1_host, const double* b1_host, int H, const double* W2_host,
                      const double* b2_host, int R, int activation, double kappa, int scalar_out) {
    BIND(ctx);
    REQUIRE(ctx->D > 0, "dks_set_mlp_model: call dks_set_background first (D unknown)");
    REQUIRE(W1_host && b1_host && W2_host && b2_host && H > 0 && R > 0, "dks_set_mlp_model: need W1, b1, W2, b2, H > 0, R > 0");
    if (H > dks::mlp::MAX_H) return fail(DKS_ERR_UNSUPPORTED, "dks_set_mlp_model: H=%d hidden units; at most %d supported", H,
                                         dks::mlp::MAX_H);
    if (R > 8) return fail(DKS_ERR_UNSUPPORTED, "dks_set_mlp_model: R=%d output units; at most 8 supported", R);
    int C = R;
    if (activation == DKS_ACT_BINARY_LOGISTIC) {
        REQUIRE(R == 1, "binary-logistic head needs R == 1 (got %d)", R);
        REQUIRE(kappa > 0, "binary-logistic head needs kappa > 0");
        C = 2;
    } else if (activation == DKS_ACT_SOFTMAX) {
        REQUIRE(R >= 2, "softmax head needs at least two output units (got %d)", R);
    } else if (activation != DKS_ACT_IDENTITY) {
        return fail(DKS_ERR_INVALID, "dks_set_mlp_model: unknown activation %d", activation);
    }
    ctx->C = C; ctx->R = R; ctx->H = H; ctx->act = activation; ctx->kappa = kappa; ctx->scalar_out = scalar_out;
    ctx->h_W.assign(W1_host, W1_host + (size_t)H * ctx->D);
    ctx->h_b.assign(b1_host, b1_host + H);
    ctx->h_W2.assign(W2_host, W2_host + (size_t)R * H);
    ctx->h_b2.assign(b2_host, b2_host + R);
    // unit order of the shared-plan kernel (binary head): positive W2 first, then negative, each padded to whole chunks
    ctx->mlp_hp = 0; ctx->mlp_negmask = 0;
    ctx->h_mlp_perm.clear(); ctx->h_mlp_w2abs.clear();
    if (R == 1) {
        const int CH = dks::mlp::CHUNK;
        std::vector<int> pos, neg;
        for (int u = 0; u < H; ++u) {
            if (W2_host[u] > 0) pos.push_back(u);
            else if (W2_host[u] < 0) neg.push_back(u);
        }
        const int np = (int)(pos.size() + CH - 1) / CH * CH, nn = (int)(neg.size() + CH - 1) / CH * CH;
        const int hp = (np + nn + 15) / 16 * 16;
        if (hp >= 16 && hp <= dks::mlp::MAX_H) {
            ctx->h_mlp_perm.assign(hp, -1);
            ctx->h_mlp_w2abs.assign(hp, 0.f);
            for (size_t k = 0; k < pos.size(); ++k) { ctx->h_mlp_perm[k] = pos[k]; ctx->h_mlp_w2abs[k] = (float)W2_host[pos[k]]; }
            for (size_t k = 0; k < neg.size(); ++k) {
                ctx->h_mlp_perm[np + k] = neg[k]; ctx->h_mlp_w2abs[np + k] = (float)-W2_host[neg[k]];
            }
            for (int c = np / CH; c < (np + nn) / CH; ++c) ctx->mlp_negmask |= 1u << c;
            ctx->mlp_hp = hp;
        }
    }
    ctx->mlp = true;
    ctx->fitted = false;
    return DKS_OK;
}

int dks_set_link(dks_ctx* ctx, int link) {
    BIND(ctx);
    REQUIRE(link == DKS_LINK_IDENTITY || link == DKS_LINK_LOGIT, "dks_set_link: unknown link %d", link);
    ctx->link = link;
    ctx->fitted = false;
    return DKS_OK;
}

int dks_fit(dks_ctx* ctx) {
    BIND(ctx);
    REQUIRE(ctx->N > 0 && ctx->R > 0, "dks_fit: background and model must be set first");
    const int N = ctx->N, D = ctx->D, R = ctx->R, C = ctx->C;
    if (ctx->G == 0) {  // default: one singleton group per column (DenseData default)
        if (D > DKS_MAX_GROUPS)
            return fail(DKS_ERR_UNSUPPORTED, "D=%d ungrouped columns; this build handles at most %d groups", D, DKS_MAX_GROUPS);
        ctx->G = D;
        ctx->h_goff.resize(D + 1);
        ctx->h_gcols.resize(D);
        for (int c = 0; c <= D; ++c) ctx->h_goff[c] = c;
        for (int c = 0; c < D; ++c) ctx->h_gcols[c] = c;
    }
    const int G = ctx->G;
    if (ctx->mlp && G > 64)
        return fail(DKS_ERR_UNSUPPORTED, "dks_fit: %d groups; networks are explained over at most 64 groups", G);
    const int RW = ctx->mlp ? ctx->H : R;       // rows of the first (or only) weight matrix
    {   // every column in exactly one group
        std::vector<int> seen(D, 0);
        REQUIRE((int)ctx->h_gcols.size() == D, "groups cover %d columns but the data has %d", (int)ctx->h_gcols.size(), D);
        for (int c : ctx->h_gcols) {
            REQUIRE(c >= 0 && c < D, "group column %d out of range", c);
            REQUIRE(seen[c]++ == 0, "column %d appears in more than one group", c);
        }
    }
    TRY(dev_alloc(&ctx->d_bg, (size_t)N * D));
    TRY(dev_alloc(&ctx->d_wbg, (size_t)N));
    TRY(dev_alloc(&ctx->d_W, (size_t)RW * D));
    TRY(dev_alloc(&ctx->d_b, (size_t)RW));
    TRY(dev_alloc(&ctx->d_goff, (size_t)G + 1));
    TRY(dev_alloc(&ctx->d_gcols, (size_t)D));
    TRY(dev_alloc(&ctx->d_colmin, (size_t)D));
    TRY(dev_alloc(&ctx->d_colmax, (size_t)D));
    TRY(dev_alloc(&ctx->d_colnan, (size_t)D));
    TRY(dev_alloc(&ctx->d_BW, (size_t)N * G * RW));
    TRY(dev_alloc(&ctx->d_scores, (size_t)N * RW));
    TRY(dev_alloc(&ctx->d_Bbar, (size_t)G * R));
    TRY(dev_alloc(&ctx->d_fnull, (size_t)C));
    TRY(dev_alloc(&ctx->d_linkfnull, (size_t)C));
    TRY(dev_alloc(&ctx->d_BWs, (size_t)N * G * R));
    TRY(dev_alloc(&ctx->d_bases, (size_t)N * R));
    TRY(dev_alloc(&ctx->d_wbf, (size_t)N));
    cudaStream_t st = ctx->stream;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_bg, ctx->h_bg.data(), sizeof(double) * N * D, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_wbg, ctx->h_wbg.data(), sizeof(double) * N, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_W, ctx->h_W.data(), sizeof(double) * RW * D, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_b, ctx->h_b.data(), sizeof(double) * RW, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_goff, ctx->h_goff.data(), sizeof(int32_t) * (G + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_gcols, ctx->h_gcols.data(), sizeof(int32_t) * D, cudaMemcpyHostToDevice, st));

    ctx->scale = (ctx->act == DKS_ACT_BINARY_LOGISTIC) ? -ctx->kappa * 1.4426950408889634
               : (ctx->act == DKS_ACT_SOFTMAX) ? 1.4426950408889634 : 1.0;
    if (ctx->mlp) {
        // BW1 [N][G][H] and base1 [N][H] by the linear fit kernels with W1 in place of W; fnull by a float64 forward
        const int H = ctx->H;
        TRY(dev_alloc(&ctx->d_W2, (size_t)R * H));
        TRY(dev_alloc(&ctx->d_b2, (size_t)R));
        CUDA_TRY(cudaMemcpyAsync(ctx->d_W2, ctx->h_W2.data(), sizeof(double) * R * H, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(ctx->d_b2, ctx->h_b2.data(), sizeof(double) * R, cudaMemcpyHostToDevice, st));
        if (ctx->mlp_hp > 0) {
            TRY(dev_alloc(&ctx->d_mlp_perm, (size_t)ctx->mlp_hp));
            TRY(dev_alloc(&ctx->d_mlp_w2abs, (size_t)ctx->mlp_hp));
            CUDA_TRY(cudaMemcpyAsync(ctx->d_mlp_perm, ctx->h_mlp_perm.data(), sizeof(int) * ctx->mlp_hp, cudaMemcpyHostToDevice, st));
            CUDA_TRY(cudaMemcpyAsync(ctx->d_mlp_w2abs, ctx->h_mlp_w2abs.data(), sizeof(float) * ctx->mlp_hp,
                                     cudaMemcpyHostToDevice, st));
        }
        dks::fit_bw_kernel<<<cdiv((long long)N * G * H, 256), 256, 0, st>>>(ctx->d_bg, ctx->d_W, ctx->d_goff, ctx->d_gcols, N, D,
                                                                               G, H, ctx->d_BW);
        dks::fit_scores_kernel<<<cdiv((long long)N * H, 256), 256, 0, st>>>(ctx->d_BW, ctx->d_b, N, G, H, ctx->d_scores);
        dks::fit_colstats_kernel<<<cdiv(D, 128), 128, 0, st>>>(ctx->d_bg, N, D, ctx->d_colmin, ctx->d_colmax, ctx->d_colnan);
        dks::mlp::mlp_fnull_kernel<<<1, 32, 0, st>>>(ctx->d_scores, ctx->d_wbg, N, H, ctx->d_W2, ctx->d_b2, R, C, ctx->act,
                                                     ctx->kappa, ctx->link, ctx->d_fnull, ctx->d_linkfnull);
        ctx->launches += 4;
    } else {
    dks::fit_bw_kernel<<<cdiv((long long)N * G * R, 256), 256, 0, st>>>(ctx->d_bg, ctx->d_W, ctx->d_goff, ctx->d_gcols, N, D,
                                                                           G, R, ctx->d_BW);
    dks::fit_scores_kernel<<<cdiv((long long)N * R, 256), 256, 0, st>>>(ctx->d_BW, ctx->d_b, N, G, R, ctx->d_scores);
    dks::fit_colstats_kernel<<<cdiv(D, 128), 128, 0, st>>>(ctx->d_bg, N, D, ctx->d_colmin, ctx->d_colmax, ctx->d_colnan);
    dks::fit_fnull_kernel<<<1, 256, 0, st>>>(ctx->d_scores, ctx->d_BW, ctx->d_wbg, N, G, R, C, ctx->act, ctx->kappa,
                                              ctx->link, ctx->d_fnull, ctx->d_linkfnull, ctx->d_Bbar);
    dks::fit_scale_kernel<<<cdiv((long long)N * G * R, 256), 256, 0, st>>>(ctx->d_BW, ctx->d_scores, ctx->d_wbg, N, G, R,
                                                                              ctx->scale, ctx->d_BWs, ctx->d_bases, ctx->d_wbf);
    ctx->launches += 5;
    }
    CUDA_TRY(cudaGetLastError());
    ctx->h_fnull.resize(C);
    ctx->h_linkfnull.resize(C);
    CUDA_TRY(cudaMemcpyAsync(ctx->h_fnull.data(), ctx->d_fnull, sizeof(double) * C, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(ctx->h_linkfnull.data(), ctx->d_linkfnull, sizeof(double) * C, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    ctx->cap_n = 0;  // workspace shapes depend on G, R, C
    ctx->prepared = false;
    if (any_plan_allocs(ctx)) {   // plans carry tables derived from the background/model: drop them
        free_plan_allocs(ctx, -1);
        memset(ctx->h_plans, 0, sizeof(ctx->h_plans));
        memset(ctx->h_l1, 0, sizeof(ctx->h_l1));
        ctx->max_plan_S = 0;
        CUDA_TRY(cudaMemcpy(ctx->d_plans, ctx->h_plans, sizeof(ctx->h_plans), cudaMemcpyHostToDevice));
    }
    ctx->fitted = true;
    ctx->epoch++;
    return DKS_OK;
}

int dks_num_outputs(dks_ctx* ctx, int* C) {
    BIND(ctx);
    REQUIRE(C, "dks_num_outputs: NULL");
    *C = ctx->C;
    return DKS_OK;
}

int dks_get_fnull(dks_ctx* ctx, double* fnull_host, double* expected_value_host) {
    BIND(ctx);
    REQUIRE(ctx->fitted, "dks_get_fnull: call dks_fit first");
    for (int c = 0; c < ctx->C; ++c) {
        if (fnull_host) fnull_host[c] = ctx->h_fnull[c];
        if (expected_value_host) expected_value_host[c] = ctx->h_linkfnull[c];
    }
    return DKS_OK;
}

int dks_predict_host(dks_ctx* ctx, const double* X_host, int n, double* out_host) {
    BIND(ctx);
    REQUIRE(ctx->fitted, "dks_predict_host: call dks_fit first");
    REQUIRE(X_host && out_host && n > 0, "dks_predict_host: bad arguments");
    double *dX = nullptr, *dO = nullptr;
    TRY(dev_alloc(&dX, (size_t)n * ctx->D));
    TRY(dev_alloc(&dO, (size_t)n * ctx->C));
    CUDA_TRY(cudaMemcpyAsync(dX, X_host, sizeof(double) * n * ctx->D, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->mlp)
        dks::mlp::mlp_predict_kernel<<<cdiv(n, 128), 128, 0, ctx->stream>>>(dX, ctx->d_W, ctx->d_b, ctx->d_W2, ctx->d_b2, n,
                                                                             ctx->D, ctx->H, ctx->R, ctx->C, ctx->act, ctx->kappa, dO);
    else
        dks::predict_kernel<<<cdiv(n, 128), 128, 0, ctx->stream>>>(dX, ctx->d_W, ctx->d_b, n, ctx->D, ctx->R, ctx->C, ctx->act,
                                                                    ctx->kappa, dO);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out_host, dO, sizeof(double) * n * ctx->C, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    cudaFree(dX); cudaFree(dO);
    return DKS_OK;
}

int dks_set_nsamples(dks_ctx* ctx, int nsamples) {
    BIND(ctx);
    REQUIRE(nsamples >= 0, "dks_set_nsamples: nsamples must be >= 0 (0 = auto)");
    ctx->nsamples_req = nsamples;
    return DKS_OK;
}

int dks_effective_nsamples(dks_ctx* ctx, int M, int* S) {
    REQUIRE(ctx && S && M >= 0, "dks_effective_nsamples: bad arguments");
    *S = dks_effective_S(M, ctx->nsamples_req);
    return DKS_OK;
}

int dks_set_shared_plan(dks_ctx* ctx, int M, int S, const uint64_t* zbits_host, const double* w_host) {
    BIND(ctx);
    REQUIRE(M >= 2 && M <= DKS_MAX_GROUPS, "dks_set_shared_plan: M=%d out of [2,%d]", M, DKS_MAX_GROUPS);
    REQUIRE(S >= 1 && zbits_host && w_host, "dks_set_shared_plan: bad arguments");
    uint64_t* dz = nullptr; double* dw = nullptr; double* dc = nullptr; double* di = nullptr;
    if (!ctx->plan_allocs[M].empty()) {
        // replacing the plan of this M (another nsamples): nothing in flight may still read the old buffers
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        free_plan_allocs(ctx, M);
        memset(&ctx->h_plans[M], 0, sizeof(PlanDev));
        memset(&ctx->h_l1[M], 0, sizeof(ctx->h_l1[M]));
        ctx->h_afix[M] = nullptr;
        ctx->epoch++;
    }
    const int W = dks_plan_words(M);                        // 64-bit words per coalition row
    const size_t S_even = ((size_t)S + 1) & ~(size_t)1;     // TMA bulk copies move 16-byte multiples
    CUDA_TRY(cudaMalloc((void**)&dz, sizeof(uint64_t) * S_even * W));
    CUDA_TRY(cudaMalloc((void**)&dw, sizeof(double) * S_even));
    ctx->plan_allocs[M].push_back(dz); ctx->plan_allocs[M].push_back(dw);
    CUDA_TRY(cudaMemsetAsync(dz, 0, sizeof(uint64_t) * S_even * W, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(dw, 0, sizeof(double) * S_even, ctx->stream));
    if (W <= 2) {
        CUDA_TRY(cudaMalloc((void**)&dc, sizeof(double) * (M - 1) * (M - 1)));
        ctx->plan_allocs[M].push_back(dc);
        CUDA_TRY(cudaMalloc((void**)&di, sizeof(double) * (M - 1) * (M - 1)));
        ctx->plan_allocs[M].push_back(di);
    }
    CUDA_TRY(cudaMemcpyAsync(dz, zbits_host, sizeof(uint64_t) * S * W, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(dw, w_host, sizeof(double) * S, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(ctx->d_status, 0, sizeof(int) * 2, ctx->stream));
    if (W > 2) {
        // more than 128 groups: the (M-1) x (M-1) normal matrix is factored by the host, which hands the projection over
        // with dks_set_plan_projection (the plan is not usable before)
    } else if (W == 1) {
        size_t smem = 2 * sizeof(double) * (size_t)(M - 1) * (M - 1);
        CUDA_TRY(cudaFuncSetAttribute(dks::plan_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dks::plan_factor_kernel<<<1, 256, smem, ctx->stream>>>(dz, dw, S, M, dc, di, ctx->d_status);
    } else {
        double* scratch = nullptr;
        CUDA_TRY(cudaMalloc((void**)&scratch, sizeof(double) * (M - 1) * (M - 1)));
        ctx->plan_allocs[M].push_back(scratch);
        size_t smem = sizeof(double) * (size_t)(M - 1) * (M - 1);
        CUDA_TRY(cudaFuncSetAttribute(dks::plan_factor_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dks::plan_factor_wide_kernel<<<1, 1024, smem, ctx->stream>>>(dz, dw, S, M, dc, di, scratch, ctx->d_status);
    }
    if (W <= 2) ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(ctx->h_status, ctx->d_status, sizeof(int) * 2, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (ctx->h_status[0] != 0)
        return fail(DKS_ERR_NUMERIC, "dks_set_shared_plan: normal matrix of the M=%d plan is not positive definite", M);
    PlanDev pd;
    memset(&pd, 0, sizeof(pd));
    pd.z = dz; pd.w = dw; pd.chol = dc; pd.ainv = di; pd.S = S; pd.W = W;
    pd.S_pad = (S + 31) / 32 * 32;
    if (M == ctx->G && ctx->fitted && ctx->act == DKS_ACT_BINARY_LOGISTIC && ctx->mlp) {
        // MLP contexts: the solve tables of the shared-plan path and the plan's hidden part d'(s, j) (dks_mlp.cuh)
        if (W == 1 && M - 1 <= dks::shared_path::PMAT_MAXK &&
            dks::shared_path::wls_pmat_smem(M, pd.S_pad, false) + 8192 <= (size_t)ctx->max_smem_optin) {
            float* pm = nullptr; double* dv = nullptr;
            CUDA_TRY(cudaMalloc((void**)&pm, sizeof(float) * (size_t)(M - 1) * pd.S_pad));
            CUDA_TRY(cudaMalloc((void**)&dv, sizeof(double) * (M - 1)));
            ctx->plan_allocs[M].push_back(pm); ctx->plan_allocs[M].push_back(dv);
            long long tot = (long long)(M - 1) * pd.S_pad;
            dks::shared_path::plan_pmat_kernel<<<cdiv(tot, 256), 256, 0, ctx->stream>>>(dz, dw, di, S, pd.S_pad, M, pm);
            dks::shared_path::plan_dvec_kernel<<<M - 1, 32, 0, ctx->stream>>>(dz, pm, S, pd.S_pad, M, dv);
            ctx->launches += 2;
            CUDA_TRY(cudaGetLastError());
            pd.pmat = pm; pd.dvec = dv;
        }
        const int HP = ctx->mlp_hp, N = ctx->N;
        if (HP > 0 && N <= dks::mlp::FAST_MAXN &&
            dks::mlp::shared_smem_bytes(N, HP) <= (size_t)ctx->max_smem_optin &&
            sizeof(float) * (size_t)M * HP <= (size_t)ctx->max_smem_optin) {
            float* dT = nullptr; float* ld = nullptr;
            CUDA_TRY(cudaMalloc((void**)&dT, sizeof(float) * (size_t)pd.S_pad * N * HP));
            CUDA_TRY(cudaMalloc((void**)&ld, sizeof(float) * (size_t)pd.S_pad * N));
            ctx->plan_allocs[M].push_back(dT); ctx->plan_allocs[M].push_back(ld);
            const long long tot = (long long)pd.S_pad * N * HP, tl = (long long)pd.S_pad * N;
            dks::mlp::mlp_plan_d_kernel<<<cdiv(tot, 256), 256, 0, ctx->stream>>>(dz, S, pd.S_pad, ctx->d_BW, ctx->d_scores, N, M,
                                                                                ctx->H, HP, ctx->d_mlp_perm, ctx->d_mlp_w2abs, dT);
            dks::mlp::mlp_plan_ld_kernel<<<cdiv(tl, 256), 256, 0, ctx->stream>>>(dz, S, pd.S_pad, ctx->d_BW, ctx->d_scores, N, M,
                                                                                 ctx->H, ctx->d_W2, ld);
            ctx->launches += 2;
            CUDA_TRY(cudaGetLastError());
            pd.mlp_dT = dT; pd.mlp_Ld = ld;
        }
    } else if (M == ctx->G && ctx->fitted && ctx->act == DKS_ACT_BINARY_LOGISTIC) {
        // shared-plan fast path: Dm table for the full varying set
        float* dm = nullptr;
        double* dme = nullptr;
        CUDA_TRY(cudaMalloc((void**)&dm, sizeof(float) * (size_t)ctx->N * pd.S_pad));
        CUDA_TRY(cudaMalloc((void**)&dme, sizeof(double) * (size_t)pd.S_pad));
        ctx->plan_allocs[M].push_back(dm); ctx->plan_allocs[M].push_back(dme);
        long long total = (long long)ctx->N * pd.S_pad;
        dks::shared_path::plan_dme_kernel<<<cdiv(pd.S_pad, 128), 128, 0, ctx->stream>>>(dz, W, S, pd.S_pad, ctx->d_BW, ctx->d_scores,
                                                                                       ctx->N, ctx->G, ctx->scale, dme);
        dks::shared_path::plan_dm_kernel<<<cdiv(total, 256), 256, 0, ctx->stream>>>(dz, W, S, pd.S_pad, ctx->d_BW, ctx->d_scores,
                                                                                      ctx->N, ctx->G, ctx->scale, dme, dm);
        ctx->launches += 2;
        CUDA_TRY(cudaGetLastError());
        pd.dme = dme;
        pd.dmT = dm;
        // projection form of the solve: P = inv(E^T W E) E^T W and d = P z_L
        if (W == 1 && M - 1 <= dks::shared_path::PMAT_MAXK &&
            dks::shared_path::wls_pmat_smem(M, pd.S_pad, false) + 8192 <= (size_t)ctx->max_smem_optin) {
            float* pm = nullptr; double* dv = nullptr;
            CUDA_TRY(cudaMalloc((void**)&pm, sizeof(float) * (size_t)(M - 1) * pd.S_pad));
            CUDA_TRY(cudaMalloc((void**)&dv, sizeof(double) * (M - 1)));
            ctx->plan_allocs[M].push_back(pm); ctx->plan_allocs[M].push_back(dv);
            long long tot = (long long)(M - 1) * pd.S_pad;
            dks::shared_path::plan_pmat_kernel<<<cdiv(tot, 256), 256, 0, ctx->stream>>>(dz, dw, di, S, pd.S_pad, M, pm);
            dks::shared_path::plan_dvec_kernel<<<M - 1, 32, 0, ctx->stream>>>(dz, pm, S, pd.S_pad, M, dv);
            ctx->launches += 2;
            CUDA_TRY(cudaGetLastError());
            pd.pmat = pm; pd.dvec = dv;
        }
        // float64 P, row-major per coalition, for the fused kernel (link + solve inside the coalition kernel)
        if (W == 1 && M <= 16) {
            const int kpad = dks::shared_path::fused_kpad(M);
            double* pm64 = nullptr; double* dv64 = nullptr;
            CUDA_TRY(cudaMalloc((void**)&pm64, sizeof(double) * (size_t)kpad * pd.S_pad));
            CUDA_TRY(cudaMalloc((void**)&dv64, sizeof(double) * kpad));
            ctx->plan_allocs[M].push_back(pm64); ctx->plan_allocs[M].push_back(dv64);
            long long tot = (long long)kpad * pd.S_pad;
            dks::shared_path::plan_pmat64_kernel<<<cdiv(tot, 256), 256, 0, ctx->stream>>>(dz, dw, di, S, pd.S_pad, M, kpad, pm64);
            dks::shared_path::plan_dvec64_kernel<<<kpad, 32, 0, ctx->stream>>>(dz, pm64, S, M, kpad, dv64);
            ctx->launches += 2;
            CUDA_TRY(cudaGetLastError());
            pd.pmat64 = pm64; pd.dvec64 = dv64; pd.kpad = kpad;
        }
    }
    ctx->h_plans[M] = pd;
    ctx->epoch++;
    ctx->h_afix[M] = nullptr;                       // sampling info of a replaced plan is stale
    memset(&ctx->h_sinfo[M], 0, sizeof(ctx->h_sinfo[M]));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_plans, ctx->h_plans, sizeof(ctx->h_plans), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (S > ctx->max_plan_S) ctx->max_plan_S = S;
    return DKS_OK;
}

int dks_clear_plans(dks_ctx* ctx) {
    BIND(ctx);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    free_plan_allocs(ctx, -1);
    ctx->epoch++;
    memset(ctx->h_plans, 0, sizeof(ctx->h_plans));
    memset(ctx->h_l1, 0, sizeof(ctx->h_l1));
    memset(ctx->h_afix, 0, sizeof(ctx->h_afix));
    memset(ctx->h_sinfo, 0, sizeof(ctx->h_sinfo));
    ctx->max_plan_S = 0;
    CUDA_TRY(cudaMemcpy(ctx->d_plans, ctx->h_plans, sizeof(ctx->h_plans), cudaMemcpyHostToDevice));
    return DKS_OK;
}

int dks_has_shared_plan(dks_ctx* ctx, int M, int* present) {
    REQUIRE(ctx && present && M >= 0 && M <= DKS_MAX_GROUPS, "dks_has_shared_plan: bad arguments");
    const PlanDev& pd = ctx->h_plans[M];
    *present = (pd.z != nullptr && pd.S == dks_effective_S(M, ctx->nsamples_req) && (pd.W <= 2 || pd.ptw != nullptr)) ? 1 : 0;
    return DKS_OK;
}

int dks_set_plan_projection(dks_ctx* ctx, int M, const double* pt_host, const double* dvec_host) {
    BIND(ctx);
    REQUIRE(M > 128 && M <= DKS_MAX_GROUPS, "dks_set_plan_projection: for plans of 129..%d groups (got M=%d); narrower plans "
            "are factored on the device", DKS_MAX_GROUPS, M);
    REQUIRE(pt_host && dvec_host, "dks_set_plan_projection: NULL table");
    PlanDev& pd = ctx->h_plans[M];
    REQUIRE(pd.z != nullptr && pd.W > 2, "dks_set_plan_projection: set the shared plan of M=%d first", M);
    REQUIRE(pd.ptw == nullptr, "dks_set_plan_projection: the M=%d plan already has its projection (replace the plan first)", M);
    const int nA = M - 1, kp = dks::wide::kpad(M);
    double* pt = nullptr; double* dv = nullptr;
    CUDA_TRY(cudaMalloc((void**)&pt, sizeof(double) * (size_t)pd.S_pad * kp));
    ctx->plan_allocs[M].push_back(pt);
    CUDA_TRY(cudaMalloc((void**)&dv, sizeof(double) * kp));
    ctx->plan_allocs[M].push_back(dv);
    CUDA_TRY(cudaMemsetAsync(pt, 0, sizeof(double) * (size_t)pd.S_pad * kp, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(dv, 0, sizeof(double) * kp, ctx->stream));
    // host [S][M-1] -> device [S_pad][kp] (zero padded rows and columns)
    CUDA_TRY(cudaMemcpy2DAsync(pt, sizeof(double) * kp, pt_host, sizeof(double) * nA, sizeof(double) * nA, (size_t)pd.S,
                               cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(dv, dvec_host, sizeof(double) * nA, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    pd.ptw = pt; pd.dvecw = dv; pd.kpw = kp;
    ctx->epoch++;
    CUDA_TRY(cudaMemcpy(ctx->d_plans, ctx->h_plans, sizeof(ctx->h_plans), cudaMemcpyHostToDevice));
    return DKS_OK;
}

int dks_set_l1(dks_ctx* ctx, int mode, int k, int others_plain) {
    REQUIRE(ctx && mode >= 0 && mode <= 3, "dks_set_l1: mode must be 0 (off), 1 (aic), 2 (bic) or 3 (num_features)");
    REQUIRE(mode != 3 || k >= 1, "dks_set_l1: num_features needs k >= 1");
    if (mode != ctx->l1_mode || k != ctx->l1_k || others_plain != ctx->l1_others_plain) ctx->epoch++;
    ctx->l1_mode = mode; ctx->l1_k = k; ctx->l1_others_plain = others_plain;
    return DKS_OK;
}

int dks_set_l1_tables(dks_ctx* ctx, int M, const double* gram_raw, const double* gram_norm, const double* colsum,
                      const double* scale, const double* bz, const double* gram_w, const double* b_rows,
                      const double* sqab_rows, double sum_b, double sum_sqb, int n_aug) {
    BIND(ctx);
    REQUIRE(M >= 2 && M <= DKS_MAX_GROUPS, "dks_set_l1_tables: M out of range");
    REQUIRE(gram_raw && gram_norm && colsum && scale && bz && gram_w && b_rows && sqab_rows, "dks_set_l1_tables: NULL table");
    const PlanDev& pd = ctx->h_plans[M];
    REQUIRE(pd.z != nullptr && n_aug == 2 * pd.S, "dks_set_l1_tables: set the shared plan of M=%d first (n_aug = 2 S)", M);
    const size_t mm = (size_t)M * M, S = (size_t)pd.S;
    const size_t total = 3 * mm + 3 * (size_t)M + 2 * S;
    double* base = nullptr;
    CUDA_TRY(cudaMalloc((void**)&base, sizeof(double) * total));
    ctx->plan_allocs[M].push_back(base);
    dks_ctx::L1Dev d;
    memset(&d, 0, sizeof(d));
    double* q = base;
    auto put = [&](const double* src, size_t cnt, const double** dst) -> cudaError_t {
        *dst = q;
        cudaError_t e = cudaMemcpyAsync(q, src, sizeof(double) * cnt, cudaMemcpyHostToDevice, ctx->stream);
        q += cnt;
        return e;
    };
    CUDA_TRY(put(gram_raw, mm, &d.gram_raw)); CUDA_TRY(put(gram_norm, mm, &d.gram_norm)); CUDA_TRY(put(gram_w, mm, &d.gram_w));
    CUDA_TRY(put(colsum, M, &d.colsum)); CUDA_TRY(put(scale, M, &d.scale)); CUDA_TRY(put(bz, M, &d.bz));
    CUDA_TRY(put(b_rows, S, &d.b)); CUDA_TRY(put(sqab_rows, S, &d.sqab));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    d.sum_b = sum_b; d.sum_sqb = sum_sqb; d.n_aug = n_aug; d.S = pd.S;
    ctx->h_l1[M] = d;
    ctx->epoch++;
    return DKS_OK;
}

int dks_set_plan_sampling(dks_ctx* ctx, int M, int nfixed, int n_full, int n_paired, int ncdf, const double* cdf_host,
                          double weight_left) {
    REQUIRE(ctx && M >= 2 && M <= DKS_MAX_GROUPS, "dks_set_plan_sampling: M out of range");
    REQUIRE(ncdf >= 0 && ncdf <= 32 && (ncdf == 0 || cdf_host), "dks_set_plan_sampling: at most 32 sampled subset sizes");
    REQUIRE(nfixed >= 0 && n_full >= 0 && n_paired >= 0, "dks_set_plan_sampling: bad arguments");
    DksSamplingInfo& inf = ctx->h_sinfo[M];
    memset(&inf, 0, sizeof(inf));
    inf.nfixed = nfixed; inf.n_full = n_full; inf.n_paired = n_paired; inf.ncdf = ncdf; inf.weight_left = weight_left;
    for (int k = 0; k < ncdf; ++k) inf.cdf[k] = cdf_host[k];
    // normal matrix of the enumerated prefix: the per-instance sampler adds the sampled rows' part to it
    const PlanDev& pd = ctx->h_plans[M];
    REQUIRE(pd.z != nullptr && nfixed <= pd.S, "dks_set_plan_sampling: set the shared plan of M=%d first", M);
    BIND(ctx);
    double* af = nullptr;
    CUDA_TRY(cudaMalloc((void**)&af, sizeof(double) * (M - 1) * (M - 1)));
    ctx->plan_allocs[M].push_back(af);
    dks::plan_prefix_normal_kernel<<<1, 256, sizeof(double) * (M - 1) * (M - 1), ctx->stream>>>(pd.z, pd.w, nfixed, M, af);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    ctx->h_afix[M] = af;
    // device copies of the tables the sampler reads (kept current here, not per explain call)
    if (!ctx->d_sinfo) TRY(dev_alloc(&ctx->d_sinfo, (size_t)(DKS_MAX_GROUPS + 1)));
    if (!ctx->d_afix) TRY(dev_alloc(&ctx->d_afix, (size_t)(DKS_MAX_GROUPS + 1)));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_sinfo, ctx->h_sinfo, sizeof(ctx->h_sinfo), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(ctx->d_afix, ctx->h_afix, sizeof(ctx->h_afix), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    ctx->epoch++;
    return DKS_OK;
}

int dks_set_plan_mode(dks_ctx* ctx, int mode, uint64_t seed) {
    REQUIRE(ctx && (mode == 0 || mode == 1), "dks_set_plan_mode: mode must be 0 (shared per M) or 1 (per instance, device-drawn)");
    ctx->plan_mode = mode;
    ctx->sampler_seed = seed;
    return DKS_OK;
}

int dks_set_row_offset(dks_ctx* ctx, int64_t offset) {
    REQUIRE(ctx && offset >= 0, "dks_set_row_offset: bad arguments");
    ctx->row_offset = (long long)offset;
    return DKS_OK;
}

int dks_get_instance_plans(dks_ctx* ctx, uint64_t* zbits_host, double* w_host, int* n_out, int* stride_out) {
    BIND(ctx);
    REQUIRE(n_out && stride_out, "dks_get_instance_plans: bad arguments");
    *n_out = ctx->gen_n; *stride_out = ctx->gen_stride;
    if (zbits_host && w_host && ctx->gen_n > 0) {
        const size_t cnt = (size_t)ctx->gen_n * ctx->gen_stride;
        CUDA_TRY(cudaMemcpyAsync(zbits_host, ctx->d_genz, sizeof(uint64_t) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(w_host, ctx->d_genw, sizeof(double) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    }
    return DKS_OK;
}

int dks_prepare_dev(dks_ctx* ctx, const double* X_dev, int n) {
    BIND(ctx);
    REQUIRE(ctx->fitted, "dks_prepare: call dks_fit first");
    REQUIRE(X_dev && n > 0, "dks_prepare: need X and n > 0");
    return launch_prepare(ctx, X_dev, n);
}

int dks_prepare_host(dks_ctx* ctx, const double* X_host, int n) {
    BIND(ctx);
    REQUIRE(ctx->fitted, "dks_prepare: call dks_fit first");
    REQUIRE(X_host && n > 0, "dks_prepare: need X and n > 0");
    size_t need = (size_t)n * ctx->D;
    if (need > ctx->cap_X) { TRY(dev_alloc(&ctx->d_X, need)); ctx->cap_X = need; }
    CUDA_TRY(cudaMemcpyAsync(ctx->d_X, X_host, sizeof(double) * need, cudaMemcpyHostToDevice, ctx->stream));
    return launch_prepare(ctx, ctx->d_X, n);
}

int dks_get_m_histogram(dks_ctx* ctx, int32_t* hist_host) {
    BIND(ctx);
    REQUIRE(ctx->prepared && hist_host, "dks_get_m_histogram: call dks_prepare_* first");
    CUDA_TRY(cudaMemcpyAsync(hist_host, ctx->d_hist, sizeof(int) * (ctx->G + 1), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DKS_OK;
}

int dks_get_varying(dks_ctx* ctx, int32_t* M_host, uint64_t* mask_host) {
    BIND(ctx);
    REQUIRE(ctx->prepared, "dks_get_varying: call dks_prepare_* first");
    if (M_host) CUDA_TRY(cudaMemcpyAsync(M_host, ctx->d_M, sizeof(int) * ctx->cur_n, cudaMemcpyDeviceToHost, ctx->stream));
    if (mask_host)
        CUDA_TRY(cudaMemcpyAsync(mask_host, ctx->d_vmask, sizeof(uint64_t) * ctx->cur_n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DKS_OK;
}

int dks_get_link_fx(dks_ctx* ctx, double* out_host, int n) {
    BIND(ctx);
    REQUIRE(ctx->prepared && out_host, "dks_get_link_fx: call dks_prepare_* / dks_explain_* first");
    REQUIRE(n == ctx->cur_n, "dks_get_link_fx: the last stage 1 ran over %d rows, the caller expects %d", ctx->cur_n, n);
    const size_t cnt = (size_t)ctx->cur_n * ctx->C;
    CUDA_TRY(cudaMemcpyAsync(out_host, ctx->d_dlink, sizeof(double) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < cnt; ++i) out_host[i] += ctx->h_linkfnull[i % ctx->C];   // stage 1 keeps link(f(x)) - link(fnull)
    return DKS_OK;
}

int dks_explain_dev(dks_ctx* ctx, double* phi_dev, const uint64_t* ext_zbits_dev, const double* ext_w_dev, int ext_stride) {
    BIND(ctx);
    REQUIRE(phi_dev, "dks_explain_dev: phi is NULL");
    TRY(launch_explain(ctx, phi_dev, ext_zbits_dev, ext_w_dev, ext_stride));
    return DKS_OK;
}

// after the solve: this rank's phi goes to every peer's gathered buffer (no-op without dks_set_peers)
static int launch_push(dks_ctx* ctx, const double* phi_dev) {
    if (ctx->peer_world <= 1) return DKS_OK;
    dks::PeerPush pp;
    pp.npeers = 0;
    for (int r = 0; r < ctx->peer_world; ++r) {
        double* slab = ctx->peer_base[r] + (long long)ctx->peer_rank * ctx->peer_slab;
        if (r == ctx->peer_rank && slab == phi_dev) continue;        // phi was written in place into the local slab
        pp.dst[pp.npeers++] = slab;
    }
    if (pp.npeers == 0) return DKS_OK;
    if (ctx->last_fused && ctx->push_in_kernel) {
        // the fused kernel stored its instances into the peers' buffers as it finished them: only the general kernels' rows are left
        dks::push_rows_kernel<<<8, 256, 0, ctx->stream>>>(phi_dev, pp, ctx->d_idx_other, ctx->d_counts + 1, ctx->cur_n, ctx->G, ctx->C);
        ctx->launches += 1;
        CUDA_TRY(cudaGetLastError());
        return DKS_OK;
    }
    dim3 grid(8, pp.npeers);
    dks::push_phi_kernel<<<grid, 256, 0, ctx->stream>>>(phi_dev, pp, ctx->peer_slab);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    return DKS_OK;
}

// after the pushes: signal every peer and wait for theirs (no-op without dks_set_peer_flags)
static int launch_peer_sync(dks_ctx* ctx) {
    if (ctx->peer_world <= 1 || !ctx->peer_flags_set) return DKS_OK;
    dks::PeerFlags f;
    memset(&f, 0, sizeof(f));
    f.world = ctx->peer_world; f.rank = ctx->peer_rank; f.step = ctx->d_step;
    f.mine = ctx->peer_flags[ctx->peer_rank];
    for (int r = 0; r < ctx->peer_world; ++r) f.peer[r] = ctx->peer_flags[r];
    dks::peer_sync_kernel<<<1, 32, 0, ctx->stream>>>(f, ctx->d_status);
    ctx->launches += 1;
    CUDA_TRY(cudaGetLastError());
    return DKS_OK;
}

static void drop_graph(dks_ctx* ctx) {
    if (ctx->gexec) { cudaGraphExecDestroy(ctx->gexec); ctx->gexec = nullptr; }
}

int dks_run_dev(dks_ctx* ctx, const double* X_dev, int n, double* phi_dev) {
    BIND(ctx);
    REQUIRE(ctx->fitted, "dks_run_dev: call dks_fit first");
    REQUIRE(X_dev && phi_dev && n > 0, "dks_run_dev: bad arguments");
    dks_ctx::GraphKey key{X_dev, phi_dev, n, ctx->nsamples_req, ctx->kernel_choice, ctx->plan_mode, ctx->row_offset,
                          (unsigned long long)ctx->sampler_seed, ctx->epoch, ctx->stream};
    if (ctx->graph_enabled && ctx->gexec && key == ctx->graph_key && ctx->dbg_i < 0) {
        CUDA_TRY(cudaGraphLaunch(ctx->gexec, ctx->stream));
        ctx->graph_launches++;
        ctx->launches += ctx->graph_kernels;
        ctx->last_was_graph = true;
        return DKS_OK;                          // the status word stays on the device until dks_last_status asks for it
    }
    // the second identical call is captured (the first one sized every workspace, so nothing allocates during capture)
    // (the legacy default stream cannot be captured: callers that want graph replay pass their own stream)
    const bool capturable = ctx->stream != nullptr && ctx->stream != cudaStreamLegacy && ctx->stream != cudaStreamPerThread;
    bool capture = ctx->graph_enabled && capturable && ctx->have_last_key && key == ctx->last_key && ctx->dbg_i < 0;
    ctx->last_key = key; ctx->have_last_key = true;
    if (capture) {
        drop_graph(ctx);
        if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed) != cudaSuccess) {
            cudaGetLastError();
            ctx->graph_enabled = false;          // this stream cannot be captured: plain launches from now on
            capture = false;
        } else {
            ctx->capturing = true;
        }
    }
    const int64_t launches_before = ctx->launches;
    int rc = launch_prepare(ctx, X_dev, n);
    if (rc == DKS_OK) rc = launch_explain(ctx, phi_dev, nullptr, nullptr, 0);
    if (rc == DKS_OK) rc = launch_push(ctx, phi_dev);
    if (rc == DKS_OK) rc = launch_peer_sync(ctx);
    ctx->last_was_graph = capture;          // the captured sequence runs as a graph launch below
    if (capture) {
        ctx->capturing = false;
        cudaGraph_t graph = nullptr;
        cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
        if (rc == DKS_OK && ce == cudaSuccess && graph) {
            ce = cudaGraphInstantiate(&ctx->gexec, graph, 0);
            if (ce == cudaSuccess) {
                ctx->graph_key = key;
                ctx->graph_kernels = ctx->launches - launches_before;
                ce = cudaGraphLaunch(ctx->gexec, ctx->stream);      // capturing did not execute anything
                ctx->graph_launches++;
            }
        }
        if (graph) cudaGraphDestroy(graph);
        if (rc != DKS_OK) return rc;
        if (ce != cudaSuccess) {
            drop_graph(ctx);
            cudaGetLastError();
            ctx->graph_enabled = false;                              // fall back to plain launches for good
            ctx->launches = launches_before;
            TRY(launch_prepare(ctx, X_dev, n));
            TRY(launch_explain(ctx, phi_dev, nullptr, nullptr, 0));
            TRY(launch_push(ctx, phi_dev));
            TRY(launch_peer_sync(ctx));
        }
    } else if (rc != DKS_OK) {
        return rc;
    }
    return DKS_OK;
}

int dks_set_peers(dks_ctx* ctx, int world, int rank, const uint64_t* gathered_ptrs_host, int64_t slab_doubles) {
    REQUIRE(ctx, "dks_set_peers: ctx is NULL");
    ctx->epoch++;
    if (world <= 1 || gathered_ptrs_host == nullptr) { ctx->peer_world = 0; ctx->peer_flags_set = false; return DKS_OK; }
    REQUIRE(world <= 16 && rank >= 0 && rank < world && slab_doubles > 0, "dks_set_peers: bad arguments (at most 16 ranks)");
    for (int r = 0; r < world; ++r) {
        REQUIRE(gathered_ptrs_host[r] != 0 && (gathered_ptrs_host[r] & 15) == 0, "dks_set_peers: peer buffers must be 16-byte aligned");
        ctx->peer_base[r] = reinterpret_cast<double*>(gathered_ptrs_host[r]);
    }
    REQUIRE((slab_doubles & 1) == 0, "dks_set_peers: slab size must be even (128-bit stores)");
    ctx->peer_world = world; ctx->peer_rank = rank; ctx->peer_slab = slab_doubles;
    ctx->peer_list_for = nullptr;
    return DKS_OK;
}

int dks_set_peer_flags(dks_ctx* ctx, const uint64_t* flag_ptrs_host) {
    BIND(ctx);
    ctx->epoch++;
    if (flag_ptrs_host == nullptr) { ctx->peer_flags_set = false; return DKS_OK; }
    REQUIRE(ctx->peer_world > 1, "dks_set_peer_flags: call dks_set_peers first");
    for (int r = 0; r < ctx->peer_world; ++r) {
        REQUIRE(flag_ptrs_host[r] != 0 && (flag_ptrs_host[r] & 7) == 0, "dks_set_peer_flags: flag arrays must be 8-byte aligned");
        ctx->peer_flags[r] = reinterpret_cast<unsigned long long*>(flag_ptrs_host[r]);
    }
    if (!ctx->d_step) {
        TRY(dev_alloc(&ctx->d_step, (size_t)1));
        CUDA_TRY(cudaMemset(ctx->d_step, 0, sizeof(unsigned long long)));
    }
    ctx->peer_flags_set = true;
    return DKS_OK;
}

int dks_graph_launches(dks_ctx* ctx, int64_t* count) {
    REQUIRE(ctx && count, "dks_graph_launches: bad arguments");
    *count = ctx->graph_launches;
    return DKS_OK;
}

int dks_explain_host(dks_ctx* ctx, const double* X_host, int n, double* phi_host, const uint64_t* ext_zbits_host,
                     const double* ext_w_host, int ext_stride) {
    BIND(ctx);
    REQUIRE(ctx->fitted, "dks_explain_host: call dks_fit first");
    REQUIRE(X_host && phi_host && n > 0, "dks_explain_host: bad arguments");
    TRY(dks_prepare_host(ctx, X_host, n));
    size_t need_phi = (size_t)ctx->C * n * ctx->G;
    if (need_phi > ctx->cap_phi) { TRY(dev_alloc(&ctx->d_phi, need_phi)); ctx->cap_phi = need_phi; }
    const uint64_t* dz = nullptr; const double* dw = nullptr;
    if (ext_zbits_host) {
        REQUIRE(ext_w_host && ext_stride > 0, "dks_explain_host: ext_w / ext_stride missing");
        size_t need = (size_t)n * ext_stride;
        if (need > ctx->cap_ext) { TRY(dev_alloc(&ctx->d_extz, need)); TRY(dev_alloc(&ctx->d_extw, need)); ctx->cap_ext = need; }
        CUDA_TRY(cudaMemcpyAsync(ctx->d_extz, ext_zbits_host, sizeof(uint64_t) * need, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(ctx->d_extw, ext_w_host, sizeof(double) * need, cudaMemcpyHostToDevice, ctx->stream));
        dz = ctx->d_extz; dw = ctx->d_extw;
    }
    TRY(launch_explain(ctx, ctx->d_phi, dz, dw, ext_stride));
    ctx->phi_rows = n;                      // dks_summarise_host works off this buffer
    // results travel through a pinned staging buffer: one asynchronous DMA + one host memcpy instead of the driver's
    // chunked pageable path (the caller's array is ordinary NumPy memory)
    bool direct = false;                    // the caller's array is page-locked: one DMA straight into it
    {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, phi_host) == cudaSuccess) direct = attr.type == cudaMemoryTypeHost;
        else cudaGetLastError();
    }
    if (!direct && need_phi > ctx->cap_phi_pin) {
        if (ctx->h_phi_pin) cudaFreeHost(ctx->h_phi_pin);
        ctx->h_phi_pin = nullptr; ctx->cap_phi_pin = 0;
        CUDA_TRY(cudaHostAlloc((void**)&ctx->h_phi_pin, sizeof(double) * need_phi, cudaHostAllocDefault));
        ctx->cap_phi_pin = need_phi;
    }
    CUDA_TRY(cudaMemcpyAsync(direct ? phi_host : ctx->h_phi_pin, ctx->d_phi, sizeof(double) * need_phi, cudaMemcpyDeviceToHost,
                             ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(ctx->h_status, ctx->d_status, sizeof(int) * 2, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (!direct) memcpy(phi_host, ctx->h_phi_pin, sizeof(double) * need_phi);
    return check_status(ctx);
}

int dks_summarise_host(dks_ctx* ctx, int n, const int32_t* seg_offsets_host, int Gp, double* phi_sum_host,
                       double* mean_abs_host, int32_t* order_host, int32_t* argmax_host) {
    BIND(ctx);
    REQUIRE(ctx->prepared && ctx->d_phi != nullptr && n == ctx->cur_n && n == ctx->phi_rows,
            "dks_summarise_host: the last dks_explain_host call covered %d rows, the caller expects %d", ctx->phi_rows, n);
    const int G = ctx->G, C = ctx->C;
    REQUIRE(Gp >= 1 && Gp <= G, "dks_summarise_host: Gp out of range");
    if (seg_offsets_host) {
        REQUIRE(seg_offsets_host[0] == 0 && seg_offsets_host[Gp] == G, "dks_summarise_host: segments must cover the %d groups", G);
        for (int g = 0; g < Gp; ++g) REQUIRE(seg_offsets_host[g + 1] > seg_offsets_host[g], "dks_summarise_host: empty segment");
    } else {
        REQUIRE(Gp == G, "dks_summarise_host: without segments Gp must equal the number of groups");
    }
    int* d_seg = nullptr; double* d_sum = nullptr; unsigned long long* d_abs = nullptr; double* d_mean = nullptr; int* d_ord = nullptr;
    int* d_arg = nullptr;
    const size_t cells = (size_t)C * Gp;
    TRY(dev_alloc(&d_abs, cells)); TRY(dev_alloc(&d_mean, (size_t)(C + 1) * Gp)); TRY(dev_alloc(&d_ord, (size_t)(C + 1) * Gp));
    TRY(dev_alloc(&d_arg, (size_t)n));
    if (seg_offsets_host) {
        TRY(dev_alloc(&d_seg, (size_t)Gp + 1));
        CUDA_TRY(cudaMemcpyAsync(d_seg, seg_offsets_host, sizeof(int) * (Gp + 1), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (phi_sum_host) TRY(dev_alloc(&d_sum, cells * n));
    CUDA_TRY(cudaMemsetAsync(d_abs, 0, sizeof(unsigned long long) * cells, ctx->stream));
    const long long total = (long long)cells * n;
    int grid = cdiv(total, 256);
    if (grid > ctx->sm_count * 4) grid = ctx->sm_count * 4;
    dks::phi_summary_kernel<<<grid, 256, sizeof(unsigned long long) * cells, ctx->stream>>>(
        ctx->d_phi, C, n, G, d_seg, Gp, d_sum, d_abs, ctx->d_dlink, ctx->d_linkfnull, d_arg);
    dks::phi_rank_kernel<<<1, 128, 0, ctx->stream>>>(d_abs, C, n, Gp, d_mean, d_ord);
    ctx->launches += 2;
    CUDA_TRY(cudaGetLastError());
    if (phi_sum_host) CUDA_TRY(cudaMemcpyAsync(phi_sum_host, d_sum, sizeof(double) * cells * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (mean_abs_host) CUDA_TRY(cudaMemcpyAsync(mean_abs_host, d_mean, sizeof(double) * (C + 1) * Gp, cudaMemcpyDeviceToHost, ctx->stream));
    if (order_host) CUDA_TRY(cudaMemcpyAsync(order_host, d_ord, sizeof(int) * (C + 1) * Gp, cudaMemcpyDeviceToHost, ctx->stream));
    if (argmax_host) CUDA_TRY(cudaMemcpyAsync(argmax_host, d_arg, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_abs); cudaFree(d_mean); cudaFree(d_ord); cudaFree(d_arg);
    if (d_seg) cudaFree(d_seg);
    if (d_sum) cudaFree(d_sum);
    return DKS_OK;
}

int dks_host_alloc(void** out, uint64_t bytes) {
    if (!out || bytes == 0) return fail(DKS_ERR_INVALID, "dks_host_alloc: bad arguments");
    CUDA_TRY(cudaHostAlloc(out, (size_t)bytes, cudaHostAllocDefault));
    return DKS_OK;
}

int dks_host_free(void* p) {
    if (p) CUDA_TRY(cudaFreeHost(p));
    return DKS_OK;
}

int dks_last_status(dks_ctx* ctx, int* detail) {
    BIND(ctx);
    CUDA_TRY(cudaMemcpyAsync(ctx->h_status, ctx->d_status, sizeof(int) * 2, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (detail) *detail = ctx->h_status[1];
    return check_status(ctx);
}

int dks_set_option(dks_ctx* ctx, const char* name, int value) {
    REQUIRE(ctx && name, "dks_set_option: bad arguments");
    const std::string key(name);
    if (key == "fused") ctx->opt_fused = value;
    else if (key == "fused_ni") ctx->opt_fused_ni = value;
    else if (key == "fused_warps") ctx->opt_fused_warps = value;
    else if (key == "fused_batch") ctx->opt_fused_B = value;
    else if (key == "push_in_kernel") ctx->push_in_kernel = value != 0;
    else if (key == "graph") ctx->graph_enabled = value != 0;
    else if (key == "graph_timing") ctx->opt_graph_timing = value != 0;
    else if (key == "wide_gemm") ctx->opt_wide_gemm = value == 2 ? 2 : 1;
    else if (key == "wide_acache") ctx->opt_wide_acache = value != 0;
    else return fail(DKS_ERR_INVALID, "dks_set_option: unknown option '%s'", name);
    ctx->epoch++;                      // a captured graph holds the old launch sequence
    return DKS_OK;
}

int dks_set_kernel(dks_ctx* ctx, int kernel) {
    REQUIRE(ctx && kernel >= DKS_KERNEL_AUTO && kernel <= DKS_KERNEL_SHARED, "dks_set_kernel: unknown kernel %d", kernel);
    ctx->kernel_choice = kernel;
    return DKS_OK;
}

int dks_kernel_launches(dks_ctx* ctx, int64_t* count) {
    REQUIRE(ctx && count, "dks_kernel_launches: bad arguments");
    *count = ctx->launches;
    return DKS_OK;
}

int dks_last_timings(dks_ctx* ctx, float* ms3) {
    BIND(ctx);
    REQUIRE(ms3 && ctx->prepared, "dks_last_timings: nothing to report");
    REQUIRE(ctx->timing_valid && !(ctx->last_was_graph && !ctx->opt_graph_timing),
            "dks_last_timings: the last call was a graph replay without timing nodes (dks_set_option \"graph_timing\" 1, or \"graph\" 0)");
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaEventElapsedTime(&ms3[0], ctx->ev[0], ctx->ev[1]));
    CUDA_TRY(cudaEventElapsedTime(&ms3[1], ctx->ev[2], ctx->ev[3]));
    CUDA_TRY(cudaEventElapsedTime(&ms3[2], ctx->ev[0], ctx->ev[3]));
    return DKS_OK;
}

int dks_debug_score_dump(dks_ctx* ctx, int instance) {
    REQUIRE(ctx, "null ctx");
    ctx->dbg_i = instance;
    return DKS_OK;
}

int dks_debug_get_scores(dks_ctx* ctx, float* out_host, int max_floats, int* rows, int* cols) {
    BIND(ctx);
    REQUIRE(ctx->dbg_T && out_host && rows && cols, "dks_debug_get_scores: no dump available");
    *rows = ctx->dbg_rows; *cols = ctx->dbg_cols;
    REQUIRE((long long)ctx->dbg_rows * ctx->dbg_cols <= max_floats, "dks_debug_get_scores: buffer too small");
    CUDA_TRY(cudaMemcpyAsync(out_host, ctx->dbg_T, sizeof(float) * ctx->dbg_rows * ctx->dbg_cols, cudaMemcpyDeviceToHost,
                             ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DKS_OK;
}

int dks_debug_get_timeline(dks_ctx* ctx, float* out_host /* [6][256] */) {
    BIND(ctx);
    REQUIRE(ctx->dbg_time && out_host, "dks_debug_get_timeline: no timeline available");
    CUDA_TRY(cudaMemcpyAsync(out_host, ctx->dbg_time, sizeof(float) * 6 * 256, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DKS_OK;
}

}  // extern "C"
