// Binaural cue errors on the GPU (SURVEY.md section 8 f-2, second half): the interaural level and time difference errors of
// /root/reference/src/eval/binaural.py:6-149, static (one window = the whole signal) and "moving" (250 ms windows,
// `chunk_and_mask` :6-42: C = 1 + (T-1)//FW windows, zero padding past T, a window is valid when max over ears of
// sqrt(mean(gt^2)) >= rms_threshold).
//   ILD per window  10 log10(sum l^2 / sum r^2)                                           compute_ild :44-47
//   ITD per window  argmax (first index) over k in [-t_max, t_max] of |c[k]|, c[k] = sum_n l[(n+k) mod L] r[n]
//                   -- irfft(rfft(l) conj(rfft(r))) restricted to 2 t_max + 1 lags, as direct lag sums; ITD = tau/sr*1e6
//                                                                                         axiswise_xcorr :83-92, compute_itd :94-117
//   static:  |ild_est - ild_gt|, |itd_est - itd_gt|
//   moving:  |mean_valid(ild_est) - mean_valid(ild_gt)|,  mean_valid |itd_est - itd_gt|    ild_diff :62-81, itd_diff :134-143
// Non-finite values come out as the reference's do: a silent ear gives +-inf / NaN ILD, no valid window gives NaN.
//
// bincue_partial_kernel, grid (segment, window, mixture): one CTA stages BC_SEG right-ear samples of est and gt, packed
// (est, gt) as float2, and the left ears with the +-t_max halo wrapped circularly within the window, then every thread
// accumulates J = 8 consecutive lags over a run of samples with FFMA2 (fp32 over <= BC_SEG / P samples).  The per-thread
// runs and the four energies are summed in double in a fixed order and written to the workspace.
// bincue_finish_kernel, one CTA per mixture: sums the segments of each window in order, first-index argmax, ILD, mask,
// masked means.  No atomics, so two calls give bit-identical results.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string>

#include "common.cuh"
#include "../../include/lookonce_b200.h"

namespace l2h {
int fail(int code, const std::string& msg);

constexpr int BC_THREADS = 256;
constexpr int BC_SEG = 2048;                              // right-ear samples of one window per CTA
constexpr int BC_J = 8;                                   // lags per thread
constexpr int BC_TMAX = 256;                              // largest t_max accepted (2 t_max + 1 = 513 lags)
constexpr int BC_LS = BC_SEG + 2 * BC_TMAX + 2 * BC_J;    // left-ear staging: segment + halo + overhang of the last lag group
constexpr int BC_REC = 5;                                 // per-window record: ild_est, ild_gt, itd_est, itd_gt, valid

__device__ __forceinline__ double bc_blk_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = (threadIdx.x & 31) < (blockDim.x >> 5) ? red[threadIdx.x & 31] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    return t;
}

// part[b][w][seg][2K + 4] = { c_est[K], c_gt[K], sum l_est^2, sum r_est^2, sum l_gt^2, sum r_gt^2 } over this segment
__global__ void __launch_bounds__(BC_THREADS)
bincue_partial_kernel(const float* __restrict__ est, const float* __restrict__ gt, int T, int L, int tm, int K, int G, int P,
                      int PL, double* __restrict__ part) {
    __shared__ __align__(16) float2 smem[BC_LS + BC_SEG];
    __shared__ double red[32];
    float2* ls = smem;                   // ls[i] = (est, gt) left ear at window position s0 - tm + i, circular within the window
    float2* rs = smem + BC_LS;           // rs[n] = (est, gt) right ear at window position s0 + n
    const int seg = blockIdx.x, w = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
    const int s0 = seg * BC_SEG;
    const int64_t w0 = (int64_t)w * L;   // window start in the signal; samples at or past T are the reference's zero padding
    const float* el = est + (int64_t)b * 2 * T;
    const float* gl = gt + (int64_t)b * 2 * T;
    const float* er = el + T;
    const float* gr = gl + T;
    // every load of a thread is issued before the first store, so that each thread keeps ~40 reads in flight
    constexpr int R_IT = BC_SEG / BC_THREADS, L_IT = (BC_LS + BC_THREADS - 1) / BC_THREADS;
    const int nl = K ? BC_SEG + G * BC_J : BC_SEG;          // without lags only the segment itself (tm = 0)
    float2 rstage[R_IT], lstage[L_IT];
#pragma unroll
    for (int it = 0; it < R_IT; ++it) {
        const int pos = s0 + tid + it * BC_THREADS;
        rstage[it] = (pos < L && w0 + pos < T) ? make_float2(er[w0 + pos], gr[w0 + pos]) : make_float2(0.f, 0.f);
    }
#pragma unroll
    for (int it = 0; it < L_IT; ++it) {
        const int i = tid + it * BC_THREADS;
        int pos = s0 - tm + i;
        if (pos < 0) pos += L;
        else if (pos >= L) pos -= L;                           // tm <= L/2: one wrap reaches every position paired with n < L
        lstage[it] = (i < nl && pos < L && w0 + pos < T) ? make_float2(el[w0 + pos], gl[w0 + pos]) : make_float2(0.f, 0.f);
    }
    double e_le = 0.0, e_re = 0.0, e_lg = 0.0, e_rg = 0.0;
#pragma unroll
    for (int it = 0; it < R_IT; ++it) {
        rs[tid + it * BC_THREADS] = rstage[it];
        e_re += (double)rstage[it].x * rstage[it].x;
        e_rg += (double)rstage[it].y * rstage[it].y;
    }
#pragma unroll
    for (int it = 0; it < L_IT; ++it) {
        const int i = tid + it * BC_THREADS;
        if (i < nl) ls[i] = lstage[it];
        if (i >= tm && i < tm + BC_SEG && s0 - tm + i < L) {   // the segment's own samples count towards the energy
            e_le += (double)lstage[it].x * lstage[it].x;
            e_lg += (double)lstage[it].y * lstage[it].y;
        }
    }
    __syncthreads();

    // thread (g, p): lags -tm + g J .. -tm + g J + J - 1 over samples [p PL, (p+1) PL); g runs fastest, so the lanes of a
    // warp that share p read the same rs words (broadcast)
    const int g = G ? tid % G : 0, p = G ? tid / G : P;
    const bool active = K > 0 && p < P;
    float2 acc[BC_J];
#pragma unroll
    for (int j = 0; j < BC_J; ++j) acc[j] = make_float2(0.f, 0.f);
    if (active) {
        const int n0 = p * PL;
        int n1 = min(n0 + PL, BC_SEG);
        n1 = min(n1, (L - s0 + BC_J - 1) / BC_J * BC_J);       // right-ear samples past the window end are zero
        const float2* lp = ls + g * BC_J;                       // lp[n + j] = left at position n + (lag j of this group)
        float2 lw[2 * BC_J], rv[BC_J];
#pragma unroll
        for (int j = 0; j < BC_J; j += 2) {
            const float4 q = *reinterpret_cast<const float4*>(lp + n0 + j);
            lw[j] = make_float2(q.x, q.y);
            lw[j + 1] = make_float2(q.z, q.w);
        }
        for (int n = n0; n < n1; n += BC_J) {
#pragma unroll
            for (int j = 0; j < BC_J; j += 2) {
                const float4 q = *reinterpret_cast<const float4*>(lp + n + BC_J + j);
                lw[BC_J + j] = make_float2(q.x, q.y);
                lw[BC_J + j + 1] = make_float2(q.z, q.w);
                const float4 r = *reinterpret_cast<const float4*>(rs + n + j);
                rv[j] = make_float2(r.x, r.y);
                rv[j + 1] = make_float2(r.z, r.w);
            }
#pragma unroll
            for (int m = 0; m < BC_J; ++m)
#pragma unroll
                for (int j = 0; j < BC_J; ++j) acc[j] = ffma2(lw[m + j], rv[m], acc[j]);
#pragma unroll
            for (int j = 0; j < BC_J; ++j) lw[j] = lw[BC_J + j];
        }
    }
    __syncthreads();                                            // the staging buffer now holds the per-thread partials
    float2* pr = smem;                                          // pr[p][g J + j], P G J <= BC_THREADS J float2
    const int GJ = G * BC_J;
    if (active) {
#pragma unroll
        for (int j = 0; j < BC_J; ++j) pr[p * GJ + g * BC_J + j] = acc[j];
    }
    __syncthreads();
    double* out = part + (((int64_t)b * gridDim.y + w) * gridDim.x + seg) * (2 * K + 4);
    for (int k = tid; k < K; k += BC_THREADS) {
        double se = 0.0, sg = 0.0;
        for (int q = 0; q < P; ++q) {
            const float2 v = pr[q * GJ + k];
            se += v.x;
            sg += v.y;
        }
        out[k] = se;
        out[K + k] = sg;
    }
    e_le = bc_blk_sum(e_le, red);
    e_re = bc_blk_sum(e_re, red);
    e_lg = bc_blk_sum(e_lg, red);
    e_rg = bc_blk_sum(e_rg, red);
    if (tid == 0) {
        out[2 * K + 0] = e_le;
        out[2 * K + 1] = e_re;
        out[2 * K + 2] = e_lg;
        out[2 * K + 3] = e_rg;
    }
}

__device__ __forceinline__ void bc_keep_first_max(double& best, int& bi) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
}

// first-index argmax of |c| over the K lags of one window, est and gt (sums over the S segments in order); every lane
// gets both indices
__device__ __forceinline__ void bc_warp_argmax(const double* pw, int S, int R, int K, int lane, int* tau_e, int* tau_g) {
    double be = -1.0, bg = -1.0;
    int ie = 0, ig = 0;
    for (int k = lane; k < K; k += 32) {
        double ce = 0.0, cg = 0.0;
#pragma unroll 8
        for (int s = 0; s < S; ++s) {
            ce += pw[(int64_t)s * R + k];
            cg += pw[(int64_t)s * R + K + k];
        }
        if (fabs(ce) > be) { be = fabs(ce); ie = k; }
        if (fabs(cg) > bg) { bg = fabs(cg); ig = k; }
    }
    bc_keep_first_max(be, ie);
    bc_keep_first_max(bg, ig);
    *tau_e = ie;
    *tau_g = ig;
}

__global__ void __launch_bounds__(BC_THREADS)
bincue_finish_kernel(const double* __restrict__ part, int C, int S, int L, int tm, int K, int sr, int moving, double thr,
                     double* __restrict__ rec, float* __restrict__ out, float* __restrict__ win) {
    __shared__ double red[32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int R = 2 * K + 4;
    for (int w = tid >> 5; w < C; w += BC_THREADS / 32) {
        const double* pw = part + ((int64_t)b * C + w) * S * R;
        double e = 0.0;                                          // lanes 0..3: the four energies of the window
        if (lane < 4) {
#pragma unroll 8
            for (int s = 0; s < S; ++s) e += pw[(int64_t)s * R + 2 * K + lane];
        }
        const double e_le = __shfl_sync(0xffffffffu, e, 0), e_re = __shfl_sync(0xffffffffu, e, 1);
        const double e_lg = __shfl_sync(0xffffffffu, e, 2), e_rg = __shfl_sync(0xffffffffu, e, 3);
        double itd_e = nan(""), itd_g = nan("");
        if (K) {
            int ie, ig;
            bc_warp_argmax(pw, S, R, K, lane, &ie, &ig);
            itd_e = (double)(ie - tm) / sr * 1e6;
            itd_g = (double)(ig - tm) / sr * 1e6;
        }
        if (lane == 0) {
            double* o = rec + ((int64_t)b * C + w) * BC_REC;
            o[0] = 10.0 * log10(e_le / e_re);
            o[1] = 10.0 * log10(e_lg / e_rg);
            o[2] = itd_e;
            o[3] = itd_g;
            o[4] = (!moving || sqrt(fmax(e_lg, e_rg) / L) >= thr) ? 1.0 : 0.0;
            if (win)
                for (int q = 0; q < BC_REC; ++q) win[((int64_t)b * C + w) * BC_REC + q] = (float)o[q];
        }
    }
    __syncthreads();                                            // the window records are visible to the whole CTA
    double n = 0.0, s_ie = 0.0, s_ig = 0.0, s_dt = 0.0;
    for (int w = tid; w < C; w += BC_THREADS) {
        const double* o = rec + ((int64_t)b * C + w) * BC_REC;
        if (o[4] != 0.0) {
            n += 1.0;
            s_ie += o[0];
            s_ig += o[1];
            s_dt += fabs(o[2] - o[3]);
        }
    }
    n = bc_blk_sum(n, red);
    s_ie = bc_blk_sum(s_ie, red);
    s_ig = bc_blk_sum(s_ig, red);
    s_dt = bc_blk_sum(s_dt, red);
    if (tid == 0) {                                             // n = 0: 0/0 = NaN, the mean of an empty list
        out[b * 2 + 0] = (float)fabs(s_ie / n - s_ig / n);
        out[b * 2 + 1] = (float)(s_dt / n);
    }
}

struct BincueGeom {
    int L, C, S, tm, K, G, P, PL;
};

static int bincue_geometry(int32_t batch, int32_t n_samples, int32_t frame, int32_t t_max, BincueGeom* g) {
    if (batch <= 0 || batch > 65535 || n_samples <= 0 || frame < 0 || t_max < 0)
        return fail(1, "l2h_eval_binaural: bad argument");
    if (t_max > BC_TMAX)
        return fail(1, "l2h_eval_binaural: t_max = " + std::to_string(t_max) + " exceeds " + std::to_string(BC_TMAX) +
                           " lags (the reference's TMAX = round(1e-3 sr): sampling rates up to 256 kHz)");
    g->L = frame ? frame : n_samples;
    g->C = frame ? 1 + (n_samples - 1) / frame : 1;
    if (g->C > 65535) return fail(1, "l2h_eval_binaural: more than 65535 windows");
    if (t_max > 0 && (g->L & 1))
        return fail(1, "l2h_eval_binaural: ITD needs an even window length, got " + std::to_string(g->L) +
                           " (for odd lengths the reference's irfft returns L-1 samples and its 'correlation' is not one)");
    g->tm = t_max < g->L / 2 ? t_max : g->L / 2;
    g->K = g->tm > 0 ? 2 * g->tm + 1 : 0;
    g->G = (g->K + BC_J - 1) / BC_J;
    int P = g->G ? BC_THREADS / g->G : 1;
    g->PL = ((BC_SEG + P - 1) / P + BC_J - 1) / BC_J * BC_J;
    g->P = (BC_SEG + g->PL - 1) / g->PL;
    g->S = (g->L + BC_SEG - 1) / BC_SEG;
    return 0;
}

static size_t bincue_part_bytes(int32_t batch, const BincueGeom& g) {
    return sizeof(double) * (size_t)batch * g.C * g.S * (2 * g.K + 4);
}
static size_t bincue_rec_bytes(int32_t batch, const BincueGeom& g) { return sizeof(double) * (size_t)batch * g.C * BC_REC; }
}  // namespace l2h

extern "C" int l2h_eval_binaural_workspace_bytes(int32_t batch, int32_t n_samples, int32_t frame, int32_t t_max, size_t* bytes) {
    using namespace l2h;
    if (!bytes) return fail(1, "l2h_eval_binaural_workspace_bytes: bytes is NULL");
    BincueGeom g;
    if (int rc = bincue_geometry(batch, n_samples, frame, t_max, &g)) return rc;
    *bytes = bincue_part_bytes(batch, g) + bincue_rec_bytes(batch, g);
    return 0;
}

extern "C" int l2h_eval_binaural(const float* est_dev, const float* gt_dev, int32_t batch, int32_t n_samples, int32_t frame,
                                 int32_t t_max, double rms_threshold, int32_t sr, float* out_dev, float* windows_dev,
                                 void* workspace_dev, size_t workspace_bytes, void* stream) {
    using namespace l2h;
    if (!est_dev || !gt_dev || !out_dev || !workspace_dev || (t_max > 0 && sr <= 0))
        return fail(1, "l2h_eval_binaural: bad argument");
    BincueGeom g;
    if (int rc = bincue_geometry(batch, n_samples, frame, t_max, &g)) return rc;
    const size_t pb = bincue_part_bytes(batch, g);
    if (workspace_bytes < pb + bincue_rec_bytes(batch, g))
        return fail(1, "l2h_eval_binaural: workspace too small (see l2h_eval_binaural_workspace_bytes)");
    double* part = static_cast<double*>(workspace_dev);
    double* rec = reinterpret_cast<double*>(static_cast<char*>(workspace_dev) + pb);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    bincue_partial_kernel<<<dim3(g.S, g.C, batch), BC_THREADS, 0, st>>>(est_dev, gt_dev, n_samples, g.L, g.tm, g.K, g.G, g.P,
                                                                         g.PL, part);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) {
        bincue_finish_kernel<<<batch, BC_THREADS, 0, st>>>(part, g.C, g.S, g.L, g.tm, g.K, sr, frame > 0, rms_threshold, rec,
                                                           out_dev, windows_dev);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return fail(3, std::string("l2h_eval_binaural: ") + cudaGetErrorString(e));
    return 0;
}
