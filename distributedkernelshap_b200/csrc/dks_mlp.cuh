// One-hidden-layer ReLU networks (scikit-learn MLPClassifier / MLPRegressor, activation='relu'): fit, stage 1 and the
// coalition kernels.  Everything after the coalition stage (link, solve, l1 selection) is the linear engine's.
//
// Algebra (DESIGN.md 5.6): for coalition s of instance i and background row j the hidden pre-activation is
//     h(i,s,j) = a(i,s) + d(s,j),   a(i,s) = sum_k z_sk XW1_i[k],   d(s,j) = base1_j - sum_k z_sk BW1_j[k]
// (H-vectors; XW1 / BW1 / base1 are what prep / fit_bw_kernel / fit_scores_kernel compute with W1 in place of W), and
//     score(i,s,j) = b2 + sum_u W2[u] relu(h_u) = b2 + (La(i,s) + Ld(s,j) + sum_u W2[u] |h_u|) / 2
// with La = W2 . a and Ld = W2 . d.  With a'_u = |W2[u]| a_u and d'_u = |W2[u]| d_u, W2[u] |h_u| = sign(W2[u]) |a'_u + d'_u|:
// one add and one add of an absolute value per (unit, masked row).
#pragma once

#include "dks_kernels.cuh"

namespace dks {
namespace mlp {

constexpr int MAX_H = 128;          // hidden units
constexpr int CHUNK = 8;            // units of one sign per chunk of the shared-plan kernel's unit order
constexpr int FAST_MAXN = 256;      // background rows the shared-plan kernel keeps in shared memory
constexpr int GEN_THREADS = 256;

// ------------------------------------------------------------------------------------------------------
// fit and model check
// ------------------------------------------------------------------------------------------------------
// float64 forward of one row's hidden pre-activations pre[H] -> head outputs out[C]
__device__ inline void forward_from_pre(const double* pre, int H, const double* __restrict__ W2, const double* __restrict__ b2,
                                        int R, int act, double kappa, double* out) {
    double z[8];
    for (int r = 0; r < R; ++r) {
        double acc = b2[r];
        for (int u = 0; u < H; ++u) acc += W2[(size_t)r * H + u] * fmax(pre[u], 0.0);
        z[r] = acc;
    }
    head_f64(z, R, act, kappa, out);
}

// fnull[c] = sum_j w_j f(bg_j)[c] from the background pre-activations base1 [N][H]; one block
__global__ void mlp_fnull_kernel(const double* __restrict__ base1, const double* __restrict__ wbg, int N, int H,
                                 const double* __restrict__ W2, const double* __restrict__ b2, int R, int C, int act,
                                 double kappa, int link, double* __restrict__ fnull, double* __restrict__ linkfnull) {
    const int t = threadIdx.x;
    if (t >= C) return;
    double acc = 0;
    for (int j = 0; j < N; ++j) {
        double out[DKS_MAX_OUT];
        forward_from_pre(base1 + (size_t)j * H, H, W2, b2, R, act, kappa, out);
        acc += out[t] * wbg[j];
    }
    fnull[t] = acc;
    linkfnull[t] = link_f(acc, link);
}

// f(X) for n rows, float64 (model check against the Python callable)
__global__ void mlp_predict_kernel(const double* __restrict__ X, const double* __restrict__ W1, const double* __restrict__ b1,
                                   const double* __restrict__ W2, const double* __restrict__ b2, int n, int D, int H, int R,
                                   int C, int act, double kappa, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double pre[MAX_H], o[DKS_MAX_OUT];
    for (int u = 0; u < H; ++u) {
        double acc = b1[u];
        for (int c = 0; c < D; ++c) acc += X[(size_t)i * D + c] * W1[(size_t)u * D + c];
        pre[u] = acc;
    }
    forward_from_pre(pre, H, W2, b2, R, act, kappa, o);
    for (int c = 0; c < C; ++c) out[(size_t)i * C + c] = o[c];
}

// ------------------------------------------------------------------------------------------------------
// stage 1: one block per instance.  XW1[i][g][u], varying_groups(), M, lists, f(x), link(f(x)) - link(fnull)
// ------------------------------------------------------------------------------------------------------
__global__ void mlp_prep_kernel(const double* __restrict__ X, const double* __restrict__ W1, const double* __restrict__ b1,
                                const double* __restrict__ W2, const double* __restrict__ b2,
                                const double* __restrict__ bg, const int32_t* __restrict__ goff,
                                const int32_t* __restrict__ gcols, const double* __restrict__ colmin,
                                const double* __restrict__ colmax, const int* __restrict__ colnan,
                                const double* __restrict__ linkfnull, int n, int N, int D, int G, int H, int R, int C,
                                int act, double kappa, int link, double* __restrict__ XW, uint64_t* __restrict__ vmask,
                                int* __restrict__ Mcnt, double* __restrict__ dlink, int* __restrict__ hist,
                                int* __restrict__ counts, int* __restrict__ idx_full, int* __restrict__ idx_other) {
    __shared__ double s_hid[MAX_H];
    __shared__ double s_z[8];
    __shared__ unsigned char s_flag[64];
    const int i = blockIdx.x;
    const double* x = X + (size_t)i * D;
    for (int idx = threadIdx.x; idx < G * H; idx += blockDim.x) {
        const int g = idx / H, u = idx - g * H;
        double acc = 0;
        for (int c = goff[g]; c < goff[g + 1]; ++c) acc += x[gcols[c]] * W1[(size_t)u * D + gcols[c]];
        XW[((size_t)i * G + g) * H + u] = acc;
    }
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
        bool varies = false;
        for (int c = goff[g]; c < goff[g + 1]; ++c) {
            const int col = gcols[c];
            const double xv = x[col];
            if (colnan[col] || isnan(xv)) {
                if (!varies)
                    for (int j = 0; j < N && !varies; ++j) varies = !np_isclose(xv, bg[(size_t)j * D + col]);
            } else {
                varies = varies || !np_isclose(xv, colmin[col]) || !np_isclose(xv, colmax[col]);
            }
        }
        s_flag[g] = varies ? 1 : 0;
    }
    __syncthreads();                                  // XW1 of this instance is visible to the block
    for (int u = threadIdx.x; u < H; u += blockDim.x) {
        double acc = b1[u];
        for (int g = 0; g < G; ++g) acc += XW[((size_t)i * G + g) * H + u];
        s_hid[u] = fmax(acc, 0.0);
    }
    __syncthreads();
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        double acc = b2[r];
        for (int u = 0; u < H; ++u) acc += W2[(size_t)r * H + u] * s_hid[u];
        s_z[r] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t m = 0;
        int M = 0;
        for (int g = 0; g < G; ++g) if (s_flag[g]) { m |= (1ull << g); ++M; }
        vmask[i] = m;
        Mcnt[i] = M;
        atomicAdd(&hist[M], 1);
        if (M == G && M >= 2) idx_full[atomicAdd(&counts[0], 1)] = i;
        else idx_other[atomicAdd(&counts[1], 1)] = i;
        double o[DKS_MAX_OUT];
        head_f64(s_z, R, act, kappa, o);
        for (int c = 0; c < C; ++c) dlink[(size_t)i * C + c] = link_f(o[c], link) - linkfnull[c];
    }
}

// ------------------------------------------------------------------------------------------------------
// General MLP kernel: one CTA per instance (grid-stride), any plan source, any head, weighted backgrounds, any N.
// For each background row j the CTA stages D_j[k][u] = XW1_i[k][u] - BW1_j[k][u] of the varying groups; a warp then
// evaluates a coalition (lanes over hidden units): h = base1_j + sum_{k in s} D_j[k], the output units by a warp sum, the
// head, and adds w_j f into the coalition's accumulators.  Then link, and the solve helpers of the linear SIMT kernel.
// ------------------------------------------------------------------------------------------------------
// the network's tables the general kernel reads next to ExplainParams (whose XW holds XW1 [n][G][H]; R = output units)
struct GenParams {
    int H;
    const double* BW1;    // [N][G][H] grouped background contributions to the hidden pre-activations
    const double* base1;  // [N][H]    background pre-activations (b1 included)
    const double* W2;     // [R][H]
    const double* b2;     // [R]
};

struct GenSmem {
    double* acc;    // [nacc][S_cap]: background sums per coalition, then link-space y in place
    double* A;      // [63*63]
    double* rhs;    // [64]
    int* vi;        // [64]
    float* Dj;      // [Mmax][MAX_H]
    float* b1j;     // [MAX_H]
    float* W2s;     // [R][MAX_H]
};

__host__ __device__ inline int gen_nacc(int act, int C) { return act == DKS_ACT_BINARY_LOGISTIC ? 2 : C; }

__host__ __device__ inline size_t gen_smem_bytes(int S_cap, int Mmax, int R, int nacc) {
    return sizeof(double) * ((size_t)nacc * S_cap + 63 * 63 + 64) + sizeof(int) * 64 +
           sizeof(float) * ((size_t)Mmax * MAX_H + MAX_H + (size_t)R * MAX_H);
}

__global__ void __launch_bounds__(GEN_THREADS, 1) mlp_general_kernel(ExplainParams p, GenParams m) {
    extern __shared__ __align__(16) unsigned char gen_raw[];
    const int nacc = gen_nacc(p.act, p.C);
    const int Mmax = p.G < 64 ? p.G : 64;
    GenSmem sm;
    sm.acc = reinterpret_cast<double*>(gen_raw);
    sm.A = sm.acc + (size_t)nacc * p.S_cap;
    sm.rhs = sm.A + 63 * 63;
    sm.vi = reinterpret_cast<int*>(sm.rhs + 64);
    sm.Dj = reinterpret_cast<float*>(sm.vi + 64);
    sm.b1j = sm.Dj + (size_t)Mmax * MAX_H;
    sm.W2s = sm.b1j + MAX_H;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int N = p.N, G = p.G, C = p.C, H = m.H, R = p.R;
    const size_t slab = (size_t)p.n * G;
    for (int idx = tid; idx < R * MAX_H; idx += blockDim.x) {
        const int r = idx / MAX_H, u = idx - r * MAX_H;
        sm.W2s[idx] = u < H ? (float)m.W2[(size_t)r * H + u] : 0.f;
    }
    const float scale = (float)p.scale;

    const int ninst = dks_inst_count(p);
    for (int qi = blockIdx.x; qi < ninst; qi += gridDim.x) {
        const int i = dks_inst_at(p, qi);
        const int M = p.Mcnt[i];
        const uint64_t vm = p.vmask[i];
        __syncthreads();  // previous instance done with shared memory
        for (int idx = tid; idx < C * G; idx += blockDim.x) p.phi[(size_t)(idx / G) * slab + (size_t)i * G + idx % G] = 0.0;
        if (M == 0) continue;
        if (M == 1) {
            if (tid < C) {
                const int g = __ffsll((long long)vm) - 1;
                p.phi[(size_t)tid * slab + (size_t)i * G + g] = p.dlink[(size_t)i * C + tid];
            }
            continue;
        }
        const int S = dks_effective_S(M, p.S_req);
        const uint64_t* zp;
        const double* wp;
        const double* chol = nullptr;
        if (p.ext_z != nullptr) {
            zp = p.ext_z + (size_t)i * p.ext_stride;
            wp = p.ext_w + (size_t)i * p.ext_stride;
            if (p.ext_chol != nullptr) chol = p.ext_chol + (size_t)i * p.ext_fstride;
        } else {
            const PlanDev pd = p.plans[M];
            if (pd.z == nullptr || pd.S != S) {
                if (tid == 0) { if (atomicCAS(&p.status[0], 0, DKS_ERR_PLAN_MISSING) == 0) p.status[1] = M; }
                continue;
            }
            zp = pd.z; wp = pd.w; chol = pd.chol;
        }
        if (S > p.S_cap) {
            if (tid == 0) { if (atomicCAS(&p.status[0], 0, DKS_ERR_INVALID) == 0) p.status[1] = i; }
            continue;
        }
        if (tid == 0) {
            int k = 0;
            for (int g = 0; g < G; ++g) if ((vm >> g) & 1ull) sm.vi[k++] = g;
        }
        for (int idx = tid; idx < nacc * S; idx += blockDim.x) sm.acc[(idx / S) * p.S_cap + idx % S] = 0.0;

        // ---- background rows: masked-row outputs accumulated per coalition (each coalition belongs to one warp)
        for (int j = 0; j < N; ++j) {
            __syncthreads();
            const double* xw = p.XW + (size_t)i * G * H;
            const double* bw = m.BW1 + (size_t)j * G * H;
            for (int idx = tid; idx < M * MAX_H; idx += blockDim.x) {
                const int k = idx / MAX_H, u = idx - k * MAX_H;
                const int g = sm.vi[k];
                sm.Dj[idx] = u < H ? (float)(xw[(size_t)g * H + u] - bw[(size_t)g * H + u]) : 0.f;
            }
            for (int u = tid; u < MAX_H; u += blockDim.x) sm.b1j[u] = u < H ? (float)m.base1[(size_t)j * H + u] : 0.f;
            __syncthreads();
            const double wj = p.wbg[j];
            for (int s = warp; s < S; s += nwarps) {
                uint64_t z = zp[s];
                float h[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) h[q] = sm.b1j[lane + 32 * q];
                while (z) {
                    const int k = __ffsll((long long)z) - 1;
                    z &= z - 1;
                    const float* row = sm.Dj + (size_t)k * MAX_H;
#pragma unroll
                    for (int q = 0; q < 4; ++q) h[q] += row[lane + 32 * q];
                }
                float sc[8];
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    sc[r] = 0.f;
                    if (r < R) {
                        float v = 0.f;
#pragma unroll
                        for (int q = 0; q < 4; ++q) v = fmaf(sm.W2s[r * MAX_H + lane + 32 * q], fmaxf(h[q], 0.f), v);
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                        sc[r] = (float)m.b2[r] + v;
                    }
                }
                if (lane == 0) {
                    if (p.act == DKS_ACT_BINARY_LOGISTIC) {
                        float t = scale * sc[0];                // -kappa*log2(e) * score
                        t = fminf(fmaxf(t, -120.f), 120.f);
                        const float u = ex2_approx(t);
                        const float r1 = rcp_approx(1.f + u);
                        sm.acc[s] += wj * (double)r1;                        // p1
                        sm.acc[p.S_cap + s] += wj * (double)(u * r1);        // p0 = 1 - p1 without cancellation
                    } else if (p.act == DKS_ACT_SOFTMAX) {
                        float mx = sc[0];
#pragma unroll
                        for (int r = 1; r < 8; ++r) if (r < R) mx = fmaxf(mx, sc[r]);
                        float den = 0.f;
#pragma unroll
                        for (int r = 0; r < 8; ++r)
                            if (r < R) { sc[r] = ex2_approx((sc[r] - mx) * 1.4426950408889634f); den += sc[r]; }
                        const float inv = rcp_approx(den);
#pragma unroll
                        for (int r = 0; r < 8; ++r) if (r < R) sm.acc[(size_t)r * p.S_cap + s] += wj * (double)(sc[r] * inv);
                    } else {
#pragma unroll
                        for (int r = 0; r < 8; ++r) if (r < R) sm.acc[(size_t)r * p.S_cap + s] += wj * (double)sc[r];
                    }
                }
            }
        }
        __syncthreads();
        // ---- link-space y per coalition and output, in place
        for (int s = tid; s < S; s += blockDim.x) {
            if (p.act == DKS_ACT_BINARY_LOGISTIC) {
                const double e1 = sm.acc[s], e0 = sm.acc[p.S_cap + s];
                sm.acc[s] = p.link == DKS_LINK_LOGIT ? log(e1 / e0) - p.linkfnull[1] : e1 - p.fnull[1];
            } else {
                double y[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    y[c] = 0.0;
                    if (c >= C) continue;
                    const double e = sm.acc[(size_t)c * p.S_cap + s];
                    if (p.link == DKS_LINK_LOGIT) {
                        double rest;
                        if (p.act == DKS_ACT_SOFTMAX) {       // 1 - ey_c as the sum of the other classes: no cancellation
                            rest = 0.0;
                            for (int c2 = 0; c2 < C; ++c2) if (c2 != c) rest += sm.acc[(size_t)c2 * p.S_cap + s];
                        } else {
                            rest = 1.0 - e;
                        }
                        y[c] = log(e / rest) - p.linkfnull[c];
                    } else {
                        y[c] = e - p.fnull[c];
                    }
                }
#pragma unroll
                for (int c = 0; c < 8; ++c) if (c < C) sm.acc[(size_t)c * p.S_cap + s] = y[c];
            }
        }
        // ---- constrained WLS per output (binary head: output 0 is the exact negation of output 1)
        if (chol != nullptr) {
            for (int idx = tid; idx < (M - 1) * (M - 1); idx += blockDim.x) sm.A[idx] = chol[idx];
        } else {
            wls_build_normal(zp, wp, S, M, sm.A, warp, nwarps);
            __syncthreads();
            if (tid < 32) {
                const bool ok = wls_cholesky_warp(sm.A, M - 1);
                if (!ok && tid == 0) { if (atomicCAS(&p.status[0], 0, DKS_ERR_NUMERIC) == 0) p.status[1] = i; }
            }
        }
        const bool binary = p.act == DKS_ACT_BINARY_LOGISTIC;
        for (int c = binary ? 1 : 0; c < C; ++c) {
            __syncthreads();
            const double delta = p.dlink[(size_t)i * C + c];
            const double* ys = sm.acc + (binary ? 0 : (size_t)c * p.S_cap);
            wls_build_rhs(zp, wp, ys, S, M, delta, sm.rhs, warp, nwarps);
            __syncthreads();
            if (tid == 0) {
                wls_solve_write(sm.A, sm.rhs, M, delta, sm.vi, p.phi + (size_t)c * slab + (size_t)i * G, 1.0);
                if (binary) {
                    double* phi0 = p.phi + (size_t)i * G;
                    const double* phi1 = p.phi + slab + (size_t)i * G;
                    for (int k = 0; k < M; ++k) { const double v = phi1[sm.vi[k]]; phi0[sm.vi[k]] = (v == 0.0) ? 0.0 : -v; }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// Shared-plan MLP kernel (binary head, uniform background weights, instances whose groups all vary).
// Hidden units are reordered (positive W2 first, then negative, each padded to a multiple of CHUNK with zero units) and
// scaled by |W2|: HP = padded count.  Per plan (dks_set_shared_plan): dT[s][j][u] = d'_u(s, j) and Ld[s][j].  Per call,
// in chunks of QC instances: mlp_atab_kernel writes a'(q, s, u) for the chunk; mlp_shared_kernel (one CTA per coalition,
// its d' tile in shared memory, one thread per instance with a' in registers) writes (sum_j p1, sum_j p0) to the
// [n][S_pad] buffer the linear shared-plan solve kernels read.
// ------------------------------------------------------------------------------------------------------
struct SharedParams {
    int N, G, H, HP, S, S_pad, QC, q0;
    double scale;             // -kappa * log2(e)
    double b2;
    unsigned negmask;         // bit c: chunk c of the unit order has negative W2
    const float* dT;          // [S_pad][N][HP]
    const float* Ld;          // [S_pad][N]
    const uint64_t* z;        // [S] plan rows
    const double* XW;         // [n][G][H] XW1 of the instances
    const int* perm;          // [HP] unit order (-1: padding)
    const float* w2abs;       // [HP] |W2| in that order (0: padding)
    float* atab;              // [QC][S_pad][HP]
    const int* list;          // instances whose groups all vary ...
    const int* count;         // ... and how many
    float2* sums;             // [n][S_pad]
};

// plan tables: dT[s][j][u] = |W2[perm u]| (base1_j - sum_k z_sk BW1_j[k])[perm u], Ld[s][j] = W2 . d(s, j)
__global__ void mlp_plan_d_kernel(const uint64_t* __restrict__ z, int S, int S_pad, const double* __restrict__ BW1,
                                  const double* __restrict__ base1, int N, int G, int H, int HP, const int* __restrict__ perm,
                                  const float* __restrict__ w2abs, float* __restrict__ dT) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)S_pad * N * HP) return;
    const int u = (int)(idx % HP);
    const long long sj = idx / HP;
    const int j = (int)(sj % N), s = (int)(sj / N);
    const int pu = perm[u];
    float v = 0.f;
    if (s < S && pu >= 0) {
        double d = base1[(size_t)j * H + pu];
        uint64_t zz = z[s];
        while (zz) {
            const int k = __ffsll((long long)zz) - 1;
            zz &= zz - 1;
            d -= BW1[((size_t)j * G + k) * H + pu];
        }
        v = (float)((double)w2abs[u] * d);
    }
    dT[idx] = v;
}

__global__ void mlp_plan_ld_kernel(const uint64_t* __restrict__ z, int S, int S_pad, const double* __restrict__ BW1,
                                   const double* __restrict__ base1, int N, int G, int H, const double* __restrict__ W2,
                                   float* __restrict__ Ld) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)S_pad * N) return;
    const int j = (int)(idx % N), s = (int)(idx / N);
    double acc = 0.0;
    if (s < S) {
        const uint64_t zs = z[s];
        for (int u = 0; u < H; ++u) {
            double d = base1[(size_t)j * H + u];
            for (int k = 0; k < G; ++k) if ((zs >> k) & 1ull) d -= BW1[((size_t)j * G + k) * H + u];
            acc += W2[u] * d;
        }
    }
    Ld[idx] = (float)acc;
}

// a'(q, s, u) = |W2[perm u]| sum_k z_sk XW1_i[k][perm u] for the chunk's instances; one CTA per instance
__global__ void __launch_bounds__(256) mlp_atab_kernel(SharedParams p) {
    extern __shared__ __align__(16) float4 at_raw[];
    float* sX = reinterpret_cast<float*>(at_raw);        // [G][HP]
    const int cnt = min(*p.count - p.q0, p.QC);
    const int q = blockIdx.x;
    if (q >= cnt) return;
    const int i = p.list[p.q0 + q];
    const int G = p.G, H = p.H, HP = p.HP, H4 = HP / 4;
    for (int idx = threadIdx.x; idx < G * HP; idx += blockDim.x) {
        const int k = idx / HP, u = idx - k * HP;
        const int pu = p.perm[u];
        sX[idx] = pu >= 0 ? (float)((double)p.w2abs[u] * p.XW[((size_t)i * G + k) * H + pu]) : 0.f;
    }
    __syncthreads();
    const float4* sX4 = reinterpret_cast<const float4*>(sX);
    float4* out = reinterpret_cast<float4*>(p.atab + (size_t)q * p.S_pad * HP);
    for (int idx = threadIdx.x; idx < p.S * H4; idx += blockDim.x) {
        const int s = idx / H4, u4 = idx - s * H4;
        uint64_t zz = p.z[s];
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        while (zz) {
            const int k = __ffsll((long long)zz) - 1;
            zz &= zz - 1;
            const float4 v = sX4[k * H4 + u4];
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        out[idx] = a;
    }
}

inline size_t shared_smem_bytes(int N, int HP) { return sizeof(float) * ((size_t)N * HP + N); }

// Lane-operations per (unit, masked row) of the inner loop as built: one FADD (a' + d') and one FADD of |.| (a partial sum)
constexpr int LANE_OPS_PER_PAIR = 2;

template <int HP>
__global__ void __launch_bounds__(128) mlp_shared_kernel(SharedParams p) {
    extern __shared__ __align__(16) float4 sh_raw[];
    float* sD = reinterpret_cast<float*>(sh_raw);        // [N][HP]
    float* sC = sD + (size_t)p.N * HP;                    // [N] scale * (b2 + Ld / 2)
    const int s = blockIdx.x, N = p.N;
    const int cnt = min(*p.count - p.q0, p.QC);
    if (cnt <= 0) return;
    {
        const float4* src = reinterpret_cast<const float4*>(p.dT + (size_t)s * N * HP);
        float4* dst = reinterpret_cast<float4*>(sD);
        for (int idx = threadIdx.x; idx < N * HP / 4; idx += blockDim.x) dst[idx] = src[idx];
        for (int j = threadIdx.x; j < N; j += blockDim.x)
            sC[j] = (float)(p.scale * (p.b2 + 0.5 * (double)p.Ld[(size_t)s * N + j]));
    }
    __syncthreads();
    constexpr int NCH = HP / CHUNK;
    const float hs = 0.5f * (float)p.scale;
    float coef[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) coef[c] = ((p.negmask >> c) & 1u) ? -hs : hs;
    for (int q = threadIdx.x; q < cnt; q += blockDim.x) {
        float a[HP];
        const float4* src = reinterpret_cast<const float4*>(p.atab + ((size_t)q * p.S_pad + s) * HP);
#pragma unroll
        for (int u4 = 0; u4 < HP / 4; ++u4) {
            const float4 v = __ldg(src + u4);
            a[4 * u4] = v.x; a[4 * u4 + 1] = v.y; a[4 * u4 + 2] = v.z; a[4 * u4 + 3] = v.w;
        }
        float ci = 0.f;                                    // scale * La / 2
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            float t = 0.f;
#pragma unroll
            for (int u = 0; u < CHUNK; ++u) t += a[c * CHUNK + u];
            ci = fmaf(coef[c], t, ci);
        }
        float acc1 = 0.f, acc0 = 0.f;
        for (int j = 0; j < N; ++j) {
            const float4* d4 = reinterpret_cast<const float4*>(sD + (size_t)j * HP);
            float t = ci + sC[j];
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                const float4 d0 = d4[2 * c], d1 = d4[2 * c + 1];
                const float* ac = a + c * CHUNK;
                const float e0 = fabsf(ac[0] + d0.x) + fabsf(ac[1] + d0.y);
                const float e1 = fabsf(ac[2] + d0.z) + fabsf(ac[3] + d0.w);
                const float e2 = fabsf(ac[4] + d1.x) + fabsf(ac[5] + d1.y);
                const float e3 = fabsf(ac[6] + d1.z) + fabsf(ac[7] + d1.w);
                t = fmaf(coef[c], (e0 + e1) + (e2 + e3), t);
            }
            t = fminf(fmaxf(t, -120.f), 120.f);
            const float u = ex2_approx(t);                 // exp(-kappa * score)
            const float r = rcp_approx(1.f + u);           // p1
            acc1 += r;
            acc0 = fmaf(u, r, acc0);                       // p0 = 1 - p1 without cancellation
        }
        p.sums[(size_t)p.list[p.q0 + q] * p.S_pad + s] = make_float2(acc1, acc0);
    }
}

}  // namespace mlp
}  // namespace dks
