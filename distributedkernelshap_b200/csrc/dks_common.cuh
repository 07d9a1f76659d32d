// Shared declarations of the B200 KernelSHAP engine (host context + device parameter blocks).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "dks.h"

#define DKS_MAX_GROUPS 1024 // coalition rows: one 64-bit word up to 64 groups; two words up to 128 and sixteen up to 1024 on
                            // the shared-plan path only
#define DKS_MAX_OUT 128     // model outputs a thread may hold in local arrays (R <= 8 score rows, C <= 8 outputs today)

// 64-bit words per coalition row of a plan over M groups: the kernels exist for rows of 1, 2 and 16 words
__host__ __device__ __forceinline__ int dks_plan_words(int M) { return M <= 64 ? 1 : (M <= 128 ? 2 : 16); }

// ---- device-visible plan table entry: one shared coalition plan per number of varying groups M ----------
struct PlanDev {
    const uint64_t* z;   // [S][W] coalition bits in upstream row order (W = dks_plan_words(M))
    const double* w;     // [S] kernel weights
    const double* chol;  // [(M-1) x (M-1)] lower Cholesky factor of E^T W E (row-major), NULL if not factored
    const double* ainv;  // [(M-1) x (M-1)] inverse of E^T W E (row-major), NULL if not computed
    const float* dmT;    // [N][S_pad] 2^(scaled background part of the score - dme[s]) for the full varying set (shared fast path)
    const double* dme;   // [S_pad] row exponents: Dm rows are normalised so that their largest entry is ~1
    const float* pmat;   // [(M-1)][S_pad] P = inv(E^T W E) E^T W (float32): beta = P y - delta * dvec
    const double* dvec;  // [(M-1)] P z_L
    const double* pmat64;  // [S_pad][kpad] float64 P, one row per coalition (fused kernel), NULL if not built
    const double* dvec64;  // [kpad] P z_L with the float64 P
    const double* ptw;     // [S_pad][kpw] float64 P^T supplied by the host for plans of more than 128 groups (dks_wide.cuh)
    const double* dvecw;   // [kpw] P z_L
    const float* mlp_dT;   // [S_pad][N][HP] |W2|-scaled hidden part d'(s, j) of the full varying set (MLP shared-plan kernel)
    const float* mlp_Ld;   // [S_pad][N] W2 . d(s, j)
    int kpw;
    int kpad;
    int S;
    int S_pad;
    int W;               // 64-bit words per row
};

// What the device-side sampler needs to continue a plan past its enumerated prefix (per M; plan.py: sampling_info)
struct DksSamplingInfo {
    int nfixed;           // enumerated rows
    int n_full;           // fully enumerated subset sizes
    int n_paired;         // sizes whose complement has a different size
    int ncdf;             // sizes left to sample (0: the plan is fully enumerated)
    double weight_left;   // kernel mass of the sampled sizes
    double cdf[32];       // cumulative probabilities of the sampled sizes (last = 1)
};

// nsamples resolution of KernelExplainer.explain: 'auto' (req <= 0) = 2M + 2^11; capped at 2^M - 2 for M <= 30
__host__ __device__ __forceinline__ int dks_effective_S(int M, int req) {
    long long s = req > 0 ? (long long)req : 2LL * M + 2048;
    if (M <= 30) {
        long long mx = (1LL << M) - 2;
        if (s > mx) s = mx;
    }
    return (int)s;
}

// ---- parameters of the fused coalition kernel ------------------------------------------------------------
struct ExplainParams {
    int n, N, G, R, C;
    int act, link;
    int S_req;
    int S_cap;            // capacity of the per-CTA y buffer (max S any instance can need)
    double scale;         // binary head: -kappa*log2(e); applied to grouped contributions
    const float* BWs;     // [R][G][N] scaled grouped background contributions (k-major: column j contiguous)
    const float* bases;   // [R][N]   scaled background scores
    const float* wbf;     // [N]      background weights (float)
    const double* wbg;    // [N]
    const double* Bbar;   // [G][R]   weighted mean grouped background contribution (identity head)
    const double* fnull;  // [C]
    const double* linkfnull;  // [C]
    const double* XW;     // [n][G][R] grouped instance contributions (unscaled)
    const uint64_t* vmask;  // [n]
    const int* Mcnt;      // [n]
    const double* dlink;  // [n][C] link(f(x)) - link(fnull)
    const PlanDev* plans; // [DKS_MAX_GROUPS + 1]
    const uint64_t* ext_z;  // per-instance plans or NULL
    const double* ext_w;
    int ext_stride;
    const double* ext_chol;   // per-instance Cholesky factor / inverse of E^T W E prepared with the plans ([n][ext_fstride],
    const double* ext_ainv;   // compact (M-1) x (M-1) row-major), or NULL: the explain kernel builds and factors it
    int ext_fstride;
    double* phi;          // [C][n][G]
    int* status;          // [2] {code, detail}
    const int* list;      // instances this launch handles (NULL = all n) ...
    const int* count;     // ... and how many (device memory)
};

// number of instances a general kernel launch handles and the q-th of them
__device__ __forceinline__ int dks_inst_count(const ExplainParams& p) { return p.list ? *p.count : p.n; }
__device__ __forceinline__ int dks_inst_at(const ExplainParams& p, int q) { return p.list ? p.list[q] : q; }

struct dks_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    int max_smem_optin = 0;

    // problem definition
    int N = 0, D = 0, G = 0, R = 0, C = 0;
    int act = -1, link = DKS_LINK_IDENTITY, scalar_out = 0;
    double kappa = 1.0;
    bool fitted = false;
    int kernel_choice = DKS_KERNEL_AUTO;
    int nsamples_req = 0;
    bool uniform_w = true;      // background weights all equal
    float* dbg_T = nullptr;     // debug dump of the tcgen05 score tile of instance dbg_i ([dbg_rows][dbg_cols])
    int dbg_i = -1, dbg_rows = 0, dbg_cols = 0;
    float* dbg_time = nullptr;  // [6][256] clock64 timeline of CTA 0 (debug kernel variant)

    // one-hidden-layer ReLU network (dks_set_mlp_model): d_W / d_b hold W1 [H x D] / b1 [H], R = output units;
    // d_BW / d_scores hold BW1 [N][G][H] / base1 [N][H]
    bool mlp = false;
    int H = 0;
    std::vector<double> h_W2, h_b2;
    double *d_W2 = nullptr, *d_b2 = nullptr;
    // shared-plan MLP kernel (binary head): unit order (positive W2 first, then negative, padded per chunk), HP = 0 when
    // the padded width exceeds the kernel's 128 units
    int mlp_hp = 0;
    unsigned mlp_negmask = 0;
    std::vector<int> h_mlp_perm;
    std::vector<float> h_mlp_w2abs;
    int* d_mlp_perm = nullptr;
    float* d_mlp_w2abs = nullptr;
    float* d_mlp_atab = nullptr;   // [QC][S_pad][HP] a'(q, s, u) of one chunk of instances
    size_t cap_mlp_atab = 0;

    // host copies
    std::vector<double> h_bg, h_wbg, h_W, h_b;
    std::vector<int32_t> h_goff, h_gcols;

    // device, fit-time
    double *d_bg = nullptr, *d_wbg = nullptr, *d_W = nullptr, *d_b = nullptr;
    int32_t *d_goff = nullptr, *d_gcols = nullptr;
    double *d_colmin = nullptr, *d_colmax = nullptr;
    int* d_colnan = nullptr;
    double *d_BW = nullptr, *d_scores = nullptr, *d_Bbar = nullptr, *d_fnull = nullptr, *d_linkfnull = nullptr;
    float *d_BWs = nullptr, *d_bases = nullptr, *d_wbf = nullptr;
    double scale = 1.0;
    std::vector<double> h_fnull, h_linkfnull;

    // plans
    PlanDev h_plans[DKS_MAX_GROUPS + 1];
    PlanDev* d_plans = nullptr;
    std::vector<void*> plan_allocs[DKS_MAX_GROUPS + 1];   // device buffers owned by the plan of each M (freed on replace)
    int max_plan_S = 0;
    // l1 feature selection (dks_set_l1 / dks_set_l1_tables): per-M tables on the device
    struct L1Dev {
        const double *gram_raw, *gram_norm, *colsum, *scale, *bz, *gram_w, *b, *sqab;
        double sum_b, sum_sqb;
        int n_aug, S;
    };
    L1Dev h_l1[DKS_MAX_GROUPS + 1] = {};
    int l1_mode = 0, l1_k = 0, l1_others_plain = 0;
    double* d_mom = nullptr;     // [n][2G + 4] per-instance moments of y
    size_t cap_mom = 0;
    double* d_yw = nullptr;      // [n][S_pad] link-space y of the wide (more than 128 groups) solve
    double* d_betaw = nullptr;   // [n][kpw] its coefficients before the delta term
    size_t cap_yw = 0, cap_betaw = 0;
    float* d_acache = nullptr;   // [n][S_pad] A(i, s) of sixteen-word rows, shared by the launches of the background chunks
    size_t cap_acache = 0;
    int opt_wide_gemm = 2;       // float64 product of the wide solve: 1 = first version, 2 = conflict-free 128 x 64 tiles
    bool opt_wide_acache = true; // A(i, s) computed by the first background chunk's launch only (measured: DESIGN.md 5.5)
    // per-instance plans drawn on the device (plan_mode 1)
    int plan_mode = 0;
    uint64_t sampler_seed = 0;
    long long row_offset = 0;
    DksSamplingInfo h_sinfo[DKS_MAX_GROUPS + 1];
    DksSamplingInfo* d_sinfo = nullptr;
    uint64_t* d_genz = nullptr;
    double* d_genw = nullptr;
    double* d_genchol = nullptr;
    double* d_genainv = nullptr;
    size_t cap_gen = 0, cap_genf = 0;
    const double* h_afix[DKS_MAX_GROUPS + 1] = {};   // per M: normal matrix of the enumerated prefix (device pointers)
    const double** d_afix = nullptr;
    int gen_stride = 0, gen_n = 0;

    // per-call workspace
    int cap_n = 0, cur_n = 0;
    bool prepared = false;
    double* d_X = nullptr;       // staging for host inputs
    size_t cap_X = 0;
    const double* cur_X = nullptr;
    double* d_XW = nullptr;
    double* d_XT = nullptr;      // [n][ceil(G/4)][16] nibble tables of the scaled grouped contributions (binary head)
    unsigned char* d_vflag = nullptr;
    uint64_t* d_vmask = nullptr;
    int* d_M = nullptr;
    double* d_dlink = nullptr;
    int* d_hist = nullptr;       // status[2], list counts[2], then the histogram of M [G + 1] (one allocation, one memset)
    int* d_status = nullptr;
    int* d_counts = nullptr;     // [0] instances on the shared fast path, [1] the others
    int* d_idx_full = nullptr;   // [n] instances whose varying set is all G groups
    int* d_idx_other = nullptr;  // [n] the rest
    float2* d_sums = nullptr;    // [n][S_pad] (sum p1, sum p0) of the shared fast path
    size_t cap_sums = 0;
    long long* d_acc = nullptr;  // [n][24] fixed-point partial beta of the fused kernel (zero between launches)
    int* d_done = nullptr;       // [n] row groups delivered per instance (zero between launches)
    double* d_phi = nullptr;
    size_t cap_phi = 0;
    int phi_rows = 0;             // rows of the last dks_explain_host result held in d_phi
    double* h_phi_pin = nullptr;  // pinned staging for results going to pageable host memory
    size_t cap_phi_pin = 0;
    uint64_t* d_extz = nullptr;
    double* d_extw = nullptr;
    size_t cap_ext = 0;
    int h_status[2] = {0, 0};

    // CUDA graph of the device-resident explain sequence (dks_run_dev): captured on the second identical call
    struct GraphKey {
        const void* X; void* phi; int n, nsamples, kernel, plan_mode; long long row_offset; unsigned long long seed;
        unsigned epoch; cudaStream_t stream;
        bool operator==(const GraphKey& o) const {
            return X == o.X && phi == o.phi && n == o.n && nsamples == o.nsamples && kernel == o.kernel &&
                   plan_mode == o.plan_mode && row_offset == o.row_offset && seed == o.seed && epoch == o.epoch &&
                   stream == o.stream;
        }
    };
    bool graph_enabled = true;    // DKS_GRAPH=0 disables
    bool capturing = false;
    bool have_last_key = false;
    GraphKey last_key{}, graph_key{};
    cudaGraphExec_t gexec = nullptr;
    unsigned epoch = 0;           // bumped by everything that changes what the sequence launches (fit, plans, ...)
    int64_t graph_launches = 0;
    int64_t graph_kernels = 0;    // kernels one replay of the captured graph launches

    // push all-gather over peer memory: after a device-resident explain, phi is stored into slab `peer_rank` of every
    // peer's gathered buffer (dks_set_peers)
    int peer_world = 0, peer_rank = 0;
    long long peer_slab = 0;                       // doubles per slab
    double* peer_base[16] = {};                    // device pointers to each rank's [world][slab] buffer
    unsigned long long* peer_flags[16] = {};       // rank r's flag array [world] (peer-mapped); [peer_rank] is this rank's own
    bool peer_flags_set = false;
    double** d_peer_list = nullptr;                // device copy of the peers' slab addresses for the current phi buffer
    double* peer_list_for = nullptr;               // the phi buffer d_peer_list was built for
    unsigned long long* d_step = nullptr;          // device-side step counter of the flag exchange
    bool push_in_kernel = false;                   // 1: the fused kernel's epilogue stores phi into the peers' buffers itself
                                                   // (measured slower than the separate coalesced push kernel: DESIGN.md §7)
    // tuning knobs (dks_set_option; defaults from the environment at dks_create: DKS_FUSED, DKS_FUSED_NI, ...)
    int opt_fused = 1, opt_fused_ni = 0, opt_fused_warps = 0, opt_fused_B = 0;
    bool opt_graph_timing = false;   // keep the timing event records inside a captured graph (dks_last_timings after replays)
    bool timing_valid = false, last_was_graph = false;
    bool last_fused = false;                       // the last explain ran the fused shared-plan kernel

    // the general kernel for the instances the shared-plan path does not take runs on a side stream, next to the fused kernel
    // (it is usually empty: a serialised empty launch cost 6 us per step)
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int64_t launches = 0;
};
