// b2t_tracker.cu -- kernels + C ABI (include/b200track.h) for the association branch:
// batched Kalman ops, "+1" IoU cost, thresholded exact assignment and the fused per-frame
// SORT / ByteTrack / BoT-SORT step and the fused C-BIoU step.  Compiled for sm_100a with --fmad=false (see b2t_iou.cuh).
#include <string>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "b2t_step.cuh"
#include "b2t_cbiou.cuh"
#include "../../include/b200track.h"

using namespace b2t;

// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static long long g_launches = 0;

static int fail(int code, const char* fmt, const char* a = "") {
    char buf[512];
    snprintf(buf, sizeof buf, fmt, a);
    g_err = buf;
    return code;
}
static int check_launch(const char* what) {
    g_launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        g_err = std::string(what) + ": " + cudaGetErrorString(e);
        return B2T_ECUDA;
    }
    return B2T_OK;
}
extern "C" const char* b2t_last_error(void) { return g_err.c_str(); }
extern "C" int b2t_version(void) { return 100; }
extern "C" long long b2t_launch_count(void) { return g_launches; }

// ------------------------------------------------------------------------------------------ Kalman kernels
template <class T>
__global__ void kalman_initiate_kernel(int fmt, const T* meas, T* mean, T* cov, int k) {
    const int r = lane_id() & 7;
    const int g = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 3);
    if (g >= k) return;
    T z[4];
    for (int q = 0; q < 4; ++q) z[q] = meas[(size_t)g * 4 + q];
    KRow<T> kr;
    kf_initiate<T>(kr, r, fmt, z);
    kf_store<T>(kr, mean + (size_t)g * 8, cov + (size_t)g * 64, r);
}

template <class T>
__global__ void kalman_predict_kernel(int fmt, T* mean, T* cov, const int* flags, int n, int q_f32) {
    const int r = lane_id() & 7;
    const int g = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 3);
    const bool on = g < n;
    KRow<T> kr;
    if (on) kf_load<T>(kr, mean + (size_t)g * 8, cov + (size_t)g * 64, r);
    else { kr.m = (T)0; for (int j = 0; j < 8; ++j) kr.p[j] = (T)0; }
    const bool zero_vh = on && flags && (flags[g] & B2T_FLAG_NOT_TRACKED);
    kf_predict<T>(kr, r, fmt, zero_vh, q_f32 != 0);
    if (on) kf_store<T>(kr, mean + (size_t)g * 8, cov + (size_t)g * 64, r);
}

template <class T>
__global__ void kalman_update_kernel(int fmt, T* mean, T* cov, const int* idx, const T* meas, const float* conf,
                                     const int* flags, int k) {
    const int r = lane_id() & 7;
    const int g = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 3);
    const bool on = g < k;
    const int row = on ? (idx ? idx[g] : g) : 0;
    KRow<T> kr;
    T z[4] = {(T)0, (T)0, (T)0, (T)0};
    if (on) {
        kf_load<T>(kr, mean + (size_t)row * 8, cov + (size_t)row * 64, r);
        for (int q = 0; q < 4; ++q) z[q] = meas[(size_t)g * 4 + q];
    } else {
        kr.m = (T)1;
        for (int j = 0; j < 8; ++j) kr.p[j] = (j == r) ? (T)1 : (T)0;
    }
    const bool f32 = on && flags && (flags[g] & B2T_FLAG_MEAN_F32);
    const float cf = (on && conf) ? conf[g] : -1.f;
    kf_update<T>(kr, r, fmt, z, f32, cf);
    if (on) kf_store<T>(kr, mean + (size_t)row * 8, cov + (size_t)row * 64, r);
}

template <class T>
__global__ void kalman_gmc_kernel(T* mean, T* cov, int n, T a00, T a01, T tx, T a10, T a11, T ty) {
    const int r = lane_id() & 7;
    const int g = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 3);
    const bool on = g < n;
    KRow<T> kr;
    if (on) kf_load<T>(kr, mean + (size_t)g * 8, cov + (size_t)g * 64, r);
    else { kr.m = (T)0; for (int j = 0; j < 8; ++j) kr.p[j] = (T)0; }
    const T w6[6] = {a00, a01, tx, a10, a11, ty};
    kf_gmc<T>(kr, r, w6);
    if (on) kf_store<T>(kr, mean + (size_t)g * 8, cov + (size_t)g * 64, r);
}

template <class T>
__global__ void kalman_project_kernel(int fmt, const T* mean, const T* cov, const int* flags, const float* conf,
                                      T* out_mean, T* out_cov, int n) {
    const int g = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (g >= n) return;
    const T* m = mean + (size_t)g * 8;
    const T* c = cov + (size_t)g * 64;
    const bool f32 = flags && (flags[g] & B2T_FLAG_MEAN_F32);
    const float cf = conf ? conf[g] : -1.f;
    for (int a = 0; a < 4; ++a) {
        out_mean[(size_t)g * 4 + a] = m[a];
        for (int b = 0; b < 4; ++b) {
            T v = c[a * 8 + b];
            if (a == b) v = v + kf_r<T>(a, fmt, m[2], m[3], f32, cf);
            out_cov[(size_t)g * 16 + a * 4 + b] = v;
        }
    }
}

// gating_distance: one state, thread per measurement.
template <class T>
__global__ void kalman_gating_kernel(int fmt, const T* mean, const T* cov, const T* meas, int m, int only_position,
                                     int metric, T* out) {
    const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= m) return;
    const int nd = only_position ? 2 : 4;
    T S[4][4], d[4];
    for (int a = 0; a < 4; ++a) {
        for (int b = 0; b < 4; ++b) S[a][b] = cov[a * 8 + b];
        S[a][a] = S[a][a] + kf_r<T>(a, fmt, mean[2], mean[3], false, -1.f);
        d[a] = meas[(size_t)i * 4 + a] - mean[a];
    }
    T acc = (T)0;
    if (metric == 1) {
        for (int a = 0; a < nd; ++a) acc = acc + d[a] * d[a];
    } else {
        T L[4][4];
        for (int a = 0; a < nd; ++a)
            for (int b = 0; b <= a; ++b) {
                T s = S[a][b];
                for (int q = 0; q < b; ++q) s = s - L[a][q] * L[b][q];
                L[a][b] = (a == b) ? sqrt(s) : s / L[b][b];
            }
        T z[4];
        for (int a = 0; a < nd; ++a) {
            T s = d[a];
            for (int q = 0; q < a; ++q) s = s - L[a][q] * z[q];
            z[a] = s / L[a][a];
            acc = acc + z[a] * z[a];
        }
    }
    out[i] = acc;
}

// ------------------------------------------------------------------------------------------ IoU cost
// grid (col tiles of 128, row tiles of 8, batch); block 128: thread = one column, loops 8 rows.
// Row boxes are staged through shared memory; each warp writes 32 consecutive costs per row.
template <class T>
__global__ void iou_cost_kernel(const T* a, int n, const T* b, int m, T* cost, int ld, int as_distance) {
    __shared__ T rows[8 * 4];
    const int batch = (int)blockIdx.z;
    const T* ab = a + (size_t)batch * n * 4;
    const T* bb = b + (size_t)batch * m * 4;
    T* cb = cost + (size_t)batch * n * ld;
    const int r0 = (int)blockIdx.y * 8;
    const int j = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (threadIdx.x < 32) {
        const int rr = r0 + ((int)threadIdx.x >> 2);
        rows[threadIdx.x] = rr < n ? ab[(size_t)rr * 4 + (threadIdx.x & 3)] : (T)0;
    }
    __syncthreads();
    if (j >= m) return;
    T bx[4];
    for (int q = 0; q < 4; ++q) bx[q] = bb[(size_t)j * 4 + q];
    for (int k = 0; k < 8; ++k) {
        const int rr = r0 + k;
        if (rr >= n) break;
        const T iou = iou_plus1<T>(rows + 4 * k, bx);
        cb[(size_t)rr * ld + j] = as_distance ? (T)1 - iou : iou;
    }
}

// ------------------------------------------------------------------------------------------ assignment
// Dense cost -> per-row compacted (col, cost) lists at fixed stride m (one read of the matrix).
template <class T>
__global__ void lap_sparsify_kernel(const T* cost, int n, int m, int ld, T thresh, int* e_col, T* e_cost, int* row_cnt,
                                    size_t ws_stride_e, size_t ws_stride_r) {
    const int batch = (int)blockIdx.y;
    const int i = (int)blockIdx.x * num_warps() + warp_id();
    if (i >= n) return;
    const T* row = cost + ((size_t)batch * n + i) * ld;
    int* oc = e_col + batch * ws_stride_e + (size_t)i * m;
    T* ov = e_cost + batch * ws_stride_e + (size_t)i * m;
    int cnt = 0;
    for (int j0 = 0; j0 < m; j0 += 32) {
        const int j = j0 + lane_id();
        T c = (T)0;
        bool f = false;
        if (j < m) { c = row[j]; f = c < thresh; }
        const unsigned bal = __ballot_sync(B2T_FULL, f);
        if (f) { const int pos = cnt + __popc(bal & lanemask_lt()); oc[pos] = j; ov[pos] = c; }
        cnt += __popc(bal);
    }
    if (lane_id() == 0) row_cnt[batch * ws_stride_r + i] = cnt;
}

template <class T>
__global__ void lap_solve_kernel(int n, int m, T thresh, const int* e_col, const T* e_cost, const int* row_cnt,
                                 size_t ws_stride_e, size_t ws_stride_r, int* x, int* y) {
    B2T_DYN_SMEM(smem_raw);
    Arena arena(smem_raw);
    LapWork<T> w;
    w.carve(arena, n, m);
    const int batch = (int)blockIdx.x;
    LapCsr<T> g;
    g.row_start = nullptr; g.row_stride = m;
    g.s_col = nullptr; g.s_cost = nullptr; g.s_cap = 0;
    g.e_row = nullptr; g.s_row = nullptr; g.n_entries = 0;
    g.row_cnt = row_cnt + batch * ws_stride_r;
    g.e_col = e_col + batch * ws_stride_e;
    g.e_cost = e_cost + batch * ws_stride_e;
    lap_solve_cta<T>(n, m, g, thresh, w);
    for (int i = (int)threadIdx.x; i < n; i += (int)blockDim.x) x[(size_t)batch * n + i] = w.x[i];
    for (int j = (int)threadIdx.x; j < m; j += (int)blockDim.x) y[(size_t)batch * m + j] = w.y[j];
}

// ------------------------------------------------------------------------------------------ fused step
template <class T>
__global__ void __launch_bounds__(512, 1)
track_step_kernel(TrackState st, StepParams prm, const float* dets, const int* det_count, const double* warps,
                  const int* id_base, double* out, int out_rows, int* stat) {
    B2T_DYN_SMEM(smem_raw);
    track_step_cta<T>(st, prm, (int)blockIdx.x, dets, det_count, warps, id_base, out, out_rows, stat, smem_raw);
}

// C-BIoU (b2t_cbiou.cuh): its own kernel, so that the three Kalman kinds above compile exactly as before
template <class T>
__global__ void __launch_bounds__(512, 1)
cbiou_step_kernel(TrackState st, StepParams prm, const float* dets, const int* det_count, const int* id_base, double* out,
                  int out_rows, int* stat) {
    B2T_DYN_SMEM(smem_raw);
    cbiou_step_cta<T>(st, prm, (int)blockIdx.x, dets, det_count, id_base, out, out_rows, stat, smem_raw);
}

__global__ void track_reset_kernel(TrackState st) {
    const int s = (int)blockIdx.x;
    const size_t o = (size_t)s * st.cap;
    for (int k = (int)threadIdx.x; k < st.cap; k += (int)blockDim.x) {
        st.freelist[o + k] = k;
        st.tid[o + k] = 0; st.state[o + k] = 0; st.activated[o + k] = 0; st.tracklet_len[o + k] = 0;
        st.start_frame[o + k] = 0; st.frame_id[o + k] = 0; st.flags[o + k] = 0; st.removed_at[o + k] = 0;
        st.cls[o + k] = 0.f; st.score[o + k] = 0.f; st.tracked[o + k] = 0; st.lost[o + k] = 0;
    }
    if (threadIdx.x < 16) st.ctrl[(size_t)s * 16 + threadIdx.x] = (threadIdx.x == CTRL_NFREE) ? st.cap : 0;
}

template <class T>
__global__ void read_slot_kernel(TrackState st, int seq, int slot, double* out72) {
    const T* m = (const T*)st.mean + ((size_t)seq * st.cap + slot) * 8;
    const T* c = (const T*)st.cov + ((size_t)seq * st.cap + slot) * 64;
    const int t = (int)threadIdx.x;
    if (t < 8) out72[t] = (double)m[t];
    if (t < 64) out72[8 + t] = (double)c[t];
}

// One of a sequence's ordered slot lists as rows of LIST_COLS doubles: id, tlwh (from the Kalman mean, STrack.tlwh basetrack.py:183-211;
// C-BIoU: the last matched detection box), cls, score, slot, state, is_activated, tracklet_len, start_frame, frame_id.
// out[cap * LIST_COLS] = the list length.
constexpr int LIST_COLS = 13;
template <class T>
__global__ void read_list_kernel(TrackState st, int kind, int fmt, int seq, int which, double* out) {
    SeqView<T> v(st, seq);
    const int n = which == 0 ? v.ctrl[CTRL_NTRACKED] : v.ctrl[CTRL_NLOST];
    const int* list = which == 0 ? v.tracked : v.lost;
    for (int k = (int)threadIdx.x; k < n; k += (int)blockDim.x) {
        const int s = list[k];
        T box[4];
        if (kind == KIND_CBIOU) {
            const T* h = v.cov + (size_t)s * 64 + CB_HIST + 4 * ((int)v.mean[(size_t)s * 8 + CB_LEN] - 1);
            for (int q = 0; q < 4; ++q) box[q] = h[q];
        } else {
            mean_to_tlwh<T>(fmt, v.mean + (size_t)s * 8, (v.flags[s] & 1) != 0, box);
        }
        double* o = out + (size_t)k * LIST_COLS;
        o[0] = (double)v.tid[s]; o[1] = (double)box[0]; o[2] = (double)box[1]; o[3] = (double)box[2]; o[4] = (double)box[3];
        o[5] = (double)v.cls[s]; o[6] = (double)v.score[s]; o[7] = (double)s; o[8] = (double)v.state[s]; o[9] = (double)v.activated[s];
        o[10] = (double)v.tracklet_len[s]; o[11] = (double)v.start_frame[s]; o[12] = (double)v.frame_id[s];
    }
    if (threadIdx.x == 0) out[(size_t)st.cap * LIST_COLS] = (double)n;
}

// ========================================================================================== C ABI
#define DISPATCH(dtype, CALL_F32, CALL_F64)                         \
    do {                                                            \
        if ((dtype) == B2T_F32) { CALL_F32; }                       \
        else if ((dtype) == B2T_F64) { CALL_F64; }                  \
        else return fail(B2T_EINVAL, "dtype must be B2T_F32 or B2T_F64"); \
    } while (0)

static inline int groups_grid(int n) { return (n * 8 + 255) / 256; }

extern "C" int b2t_kalman_initiate(int dtype, int fmt, const void* meas, void* mean, void* cov, int k, void* stream) {
    if (k < 0 || fmt < 0 || fmt > 2) return fail(B2T_EINVAL, "b2t_kalman_initiate: bad arguments");
    if (k == 0) return B2T_OK;
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(dtype,
        B2T_LAUNCH(kalman_initiate_kernel<float>, groups_grid(k), 256, 0, s, fmt, (const float*)meas, (float*)mean, (float*)cov, k),
        B2T_LAUNCH(kalman_initiate_kernel<double>, groups_grid(k), 256, 0, s, fmt, (const double*)meas, (double*)mean, (double*)cov, k));
    return check_launch("kalman_initiate");
}

extern "C" int b2t_kalman_predict(int dtype, int fmt, void* mean, void* cov, const int* flags, int n, int q_f32, void* stream) {
    if (n < 0 || fmt < 0 || fmt > 2) return fail(B2T_EINVAL, "b2t_kalman_predict: bad arguments");
    if (n == 0) return B2T_OK;
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(dtype,
        B2T_LAUNCH(kalman_predict_kernel<float>, groups_grid(n), 256, 0, s, fmt, (float*)mean, (float*)cov, flags, n, q_f32),
        B2T_LAUNCH(kalman_predict_kernel<double>, groups_grid(n), 256, 0, s, fmt, (double*)mean, (double*)cov, flags, n, q_f32));
    return check_launch("kalman_predict");
}

extern "C" int b2t_kalman_project(int dtype, int fmt, const void* mean, const void* cov, const int* flags, const float* conf,
                                  void* out_mean, void* out_cov, int n, void* stream) {
    if (n < 0 || fmt < 0 || fmt > 2) return fail(B2T_EINVAL, "b2t_kalman_project: bad arguments");
    if (n == 0) return B2T_OK;
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(dtype,
        B2T_LAUNCH(kalman_project_kernel<float>, (n + 127) / 128, 128, 0, s, fmt, (const float*)mean, (const float*)cov, flags, conf, (float*)out_mean, (float*)out_cov, n),
        B2T_LAUNCH(kalman_project_kernel<double>, (n + 127) / 128, 128, 0, s, fmt, (const double*)mean, (const double*)cov, flags, conf, (double*)out_mean, (double*)out_cov, n));
    return check_launch("kalman_project");
}

extern "C" int b2t_kalman_update(int dtype, int fmt, void* mean, void* cov, const int* idx, const void* meas,
                                 const float* conf, const int* flags, int k, void* stream) {
    if (k < 0 || fmt < 0 || fmt > 2) return fail(B2T_EINVAL, "b2t_kalman_update: bad arguments");
    if (k == 0) return B2T_OK;
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(dtype,
        B2T_LAUNCH(kalman_update_kernel<float>, groups_grid(k), 256, 0, s, fmt, (float*)mean, (float*)cov, idx, (const float*)meas, conf, flags, k),
        B2T_LAUNCH(kalman_update_kernel<double>, groups_grid(k), 256, 0, s, fmt, (double*)mean, (double*)cov, idx, (const double*)meas, conf, flags, k));
    return check_launch("kalman_update");
}

extern "C" int b2t_kalman_gating(int dtype, int fmt, const void* mean, const void* cov, const void* meas, int m,
                                 int only_position, int metric, void* out, void* stream) {
    if (m < 0 || fmt < 0 || fmt > 2 || metric < 0 || metric > 1) return fail(B2T_EINVAL, "b2t_kalman_gating: bad arguments");
    if (m == 0) return B2T_OK;
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(dtype,
        B2T_LAUNCH(kalman_gating_kernel<float>, (m + 127) / 128, 128, 0, s, fmt, (const float*)mean, (const float*)cov, (const float*)meas, m, only_position, metric, (float*)out),
        B2T_LAUNCH(kalman_gating_kernel<double>, (m + 127) / 128, 128, 0, s, fmt, (const double*)mean, (const double*)cov, (const double*)meas, m, only_position, metric, (double*)out));
    return check_launch("kalman_gating");
}

extern "C" int b2t_gmc_apply(int dtype, void* mean, void* cov, int n, const double* w, void* stream) {
    if (n < 0 || !w) return fail(B2T_EINVAL, "b2t_gmc_apply: bad arguments");
    if (n == 0) return B2T_OK;
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(dtype,
        B2T_LAUNCH(kalman_gmc_kernel<float>, groups_grid(n), 256, 0, s, (float*)mean, (float*)cov, n, (float)w[0], (float)w[1], (float)w[2], (float)w[3], (float)w[4], (float)w[5]),
        B2T_LAUNCH(kalman_gmc_kernel<double>, groups_grid(n), 256, 0, s, (double*)mean, (double*)cov, n, w[0], w[1], w[2], w[3], w[4], w[5]));
    return check_launch("gmc_apply");
}

extern "C" int b2t_iou_cost(int dtype, const void* a, int n, const void* b, int m, void* cost, int ld, int batch,
                            int as_distance, void* stream) {
    if (n < 0 || m < 0 || batch < 0 || ld < m) return fail(B2T_EINVAL, "b2t_iou_cost: bad arguments");
    if (n == 0 || m == 0 || batch == 0) return B2T_OK;
    cudaStream_t s = (cudaStream_t)stream;
    dim3 grid((m + 127) / 128, (n + 7) / 8, batch);
    DISPATCH(dtype,
        B2T_LAUNCH(iou_cost_kernel<float>, grid, 128, 0, s, (const float*)a, n, (const float*)b, m, (float*)cost, ld, as_distance),
        B2T_LAUNCH(iou_cost_kernel<double>, grid, 128, 0, s, (const double*)a, n, (const double*)b, m, (double*)cost, ld, as_distance));
    return check_launch("iou_cost");
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static size_t lap_stride_e(int n, int m) { return align_up((size_t)n * m, 64); }
static size_t lap_stride_r(int n) { return align_up((size_t)n, 64); }

extern "C" size_t b2t_lap_workspace_bytes(int dtype, int n, int m, int batch) {
    const size_t ts = dtype == B2T_F64 ? 8 : 4;
    return (size_t)batch * (lap_stride_e(n, m) * (4 + ts) + lap_stride_r(n) * 4) + 1024;
}

template <class T>
static int lap_solve_t(const T* cost, int n, int m, int ld, double thresh, int* x, int* y, void* ws, int batch, cudaStream_t s) {
    const size_t se = lap_stride_e(n, m), sr = lap_stride_r(n);
    unsigned char* p = (unsigned char*)ws;
    p = (unsigned char*)align_up((size_t)p, 256);
    T* e_cost = (T*)p;            p += sizeof(T) * se * batch;
    int* e_col = (int*)p;         p += sizeof(int) * se * batch;
    int* row_cnt = (int*)p;
    const int wpb = 8;
    dim3 g1((n + wpb - 1) / wpb, batch);
    auto k1 = lap_sparsify_kernel<T>;
    B2T_LAUNCH(k1, g1, wpb * 32, 0, s, cost, n, m, ld, (T)thresh, e_col, e_cost, row_cnt, se, sr);
    int rc = check_launch("lap_sparsify");
    if (rc) return rc;
    ArenaSize as;
    LapWork<T>::size(as, n, m);
    const size_t smem = as.off + 16;
    if (smem > 227 * 1024) return fail(B2T_ECAPACITY, "b2t_lap_solve: n, m too large for one CTA's shared memory");
    auto k2 = lap_solve_kernel<T>;
    if (B2T_SET_SMEM(k2, smem) != 0) return fail(B2T_ECUDA, "b2t_lap_solve: cannot raise dynamic shared memory");
    B2T_LAUNCH(k2, batch, 512, smem, s, n, m, (T)thresh, (const int*)e_col, (const T*)e_cost, (const int*)row_cnt, se, sr, x, y);
    return check_launch("lap_solve");
}

extern "C" int b2t_lap_solve(int dtype, const void* cost, int n, int m, int ld, double thresh, int* x, int* y,
                             void* workspace, size_t workspace_bytes, int batch, void* stream) {
    if (n < 0 || m < 0 || batch < 0 || ld < m) return fail(B2T_EINVAL, "b2t_lap_solve: bad arguments");
    if (batch == 0) return B2T_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0 || m == 0) {
        if (n) cudaMemsetAsync(x, 0xff, sizeof(int) * (size_t)n * batch, s);
        if (m) cudaMemsetAsync(y, 0xff, sizeof(int) * (size_t)m * batch, s);
        return B2T_OK;
    }
    if (workspace_bytes < b2t_lap_workspace_bytes(dtype, n, m, batch)) return fail(B2T_EINVAL, "b2t_lap_solve: workspace too small");
    if (dtype == B2T_F32) return lap_solve_t<float>((const float*)cost, n, m, ld, thresh, x, y, workspace, batch, s);
    if (dtype == B2T_F64) return lap_solve_t<double>((const double*)cost, n, m, ld, thresh, x, y, workspace, batch, s);
    return fail(B2T_EINVAL, "dtype must be B2T_F32 or B2T_F64");
}

// ------------------------------------------------------------------------------------------ tracker object
struct b2t_tracker {
    b2t_tracker_config cfg;
    TrackState st;
    StepParams prm;
    size_t smem;
    // device staging for the *_host entry point (inside the state block)
    float* d_dets; int* d_count; double* d_warps; int* d_idbase; double* d_out; int* d_stat; double* d_slot; double* d_list;
    size_t out_rows_cap;
};

struct Layout {
    size_t off = 0;
    size_t take(size_t bytes) { off = align_up(off, 256); size_t o = off; off += bytes; return o; }
};

static void layout(const b2t_tracker_config& c, unsigned char* base, b2t_tracker* t, size_t* total) {
    Layout L;
    const size_t S = c.n_seq, cap = c.cap, ts = c.dtype == B2T_F64 ? 8 : 4;
    size_t o;
#define TAKE(field, type, count) o = L.take(sizeof(type) * (count)); if (t) t->field = (type*)(base + o)
    o = L.take(ts * S * cap * 8);  if (t) t->st.mean = base + o;
    o = L.take(ts * S * cap * 64); if (t) t->st.cov = base + o;
    TAKE(st.tid, int, S * cap); TAKE(st.state, int, S * cap); TAKE(st.activated, int, S * cap);
    TAKE(st.tracklet_len, int, S * cap); TAKE(st.start_frame, int, S * cap); TAKE(st.frame_id, int, S * cap);
    TAKE(st.flags, int, S * cap); TAKE(st.removed_at, int, S * cap);
    TAKE(st.cls, float, S * cap); TAKE(st.score, float, S * cap);
    TAKE(st.tracked, int, S * cap); TAKE(st.lost, int, S * cap); TAKE(st.freelist, int, S * cap);
    TAKE(st.ctrl, int, S * 16);
    TAKE(st.e_col, int, S * (size_t)c.ecap);
    TAKE(st.e_row, int, S * (size_t)c.ecap);
    o = L.take(ts * S * (size_t)c.ecap); if (t) t->st.e_cost = base + o;
    TAKE(d_dets, float, S * (size_t)c.dmax * 6); TAKE(d_count, int, S); TAKE(d_warps, double, S * 6);
    TAKE(d_idbase, int, S); TAKE(d_out, double, S * cap * OUT_COLS); TAKE(d_stat, int, S * STAT_WORDS);
    TAKE(d_slot, double, 72);
    TAKE(d_list, double, cap * LIST_COLS + 1);
#undef TAKE
    *total = align_up(L.off, 256);
}

static int check_cfg(const b2t_tracker_config* c) {
    if (!c) return fail(B2T_EINVAL, "null config");
    if (c->kind < 0 || c->kind > 3 || (c->kind != B2T_CBIOU && (c->fmt < 0 || c->fmt > 2)) || (c->dtype != B2T_F32 && c->dtype != B2T_F64))
        return fail(B2T_EINVAL, "b2t_tracker: bad kind / fmt / dtype");
    if (c->kind == B2T_CBIOU && c->dtype != B2T_F64)
        return fail(B2T_EINVAL, "b2t_tracker: B2T_CBIOU runs in B2T_F64 only (the reference's buffered IoU is float64 and there is no Kalman "
                                "state to shrink)");
    if (c->n_seq < 1 || c->cap < 64 || c->dmax < 1 || c->dmax > 1024 || c->cap > 4096 || c->ecap < 1)
        return fail(B2T_EINVAL, "b2t_tracker: bad n_seq / cap (64..4096) / dmax (1..1024) / ecap");
    const size_t smem = c->kind == B2T_CBIOU ? cbiou_smem_bytes(c->cap, c->dmax, 0)
                      : c->dtype == B2T_F64 ? StepSmem<double>::bytes(c->cap, c->dmax, 0) : StepSmem<float>::bytes(c->cap, c->dmax, 0);
    if (smem > 227 * 1024) return fail(B2T_ECAPACITY, "b2t_tracker: cap / dmax need more than 227 KB of shared memory per CTA");
    return B2T_OK;
}

extern "C" size_t b2t_tracker_state_bytes(const b2t_tracker_config* cfg) {
    if (check_cfg(cfg)) return 0;
    size_t total = 0;
    layout(*cfg, nullptr, nullptr, &total);
    return total;
}

extern "C" int b2t_tracker_reset(b2t_tracker* t, void* stream) {
    if (!t) return fail(B2T_EINVAL, "null tracker");
    B2T_LAUNCH(track_reset_kernel, t->cfg.n_seq, 256, 0, (cudaStream_t)stream, t->st);
    return check_launch("track_reset");
}

extern "C" int b2t_tracker_create(const b2t_tracker_config* cfg, void* state_mem, void* stream, b2t_tracker** out) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!state_mem || !out || ((size_t)state_mem & 255)) return fail(B2T_EINVAL, "b2t_tracker_create: state_mem must be 256-B aligned");
    b2t_tracker* t = new b2t_tracker();
    t->cfg = *cfg;
    size_t total;
    layout(*cfg, (unsigned char*)state_mem, t, &total);
    t->st.n_seq = cfg->n_seq; t->st.cap = cfg->cap; t->st.dmax = cfg->dmax; t->st.ecap = cfg->ecap;
    const bool cbiou = cfg->kind == B2T_CBIOU;
    t->st.esm = cbiou ? cbiou_fit_esm(cfg->cap, cfg->dmax, cfg->ecap, 227 * 1024)
              : cfg->dtype == B2T_F64 ? StepSmem<double>::fit_esm(cfg->cap, cfg->dmax, cfg->ecap, 227 * 1024)
                                      : StepSmem<float>::fit_esm(cfg->cap, cfg->dmax, cfg->ecap, 227 * 1024);
    t->out_rows_cap = cfg->cap;
    StepParams& p = t->prm;
    p.kind = cfg->kind; p.fmt = cfg->fmt;
    // The reference evaluates its thresholds in Python floats (float64) and NumPy 2 then compares
    // float32 scores against them in float32 (oracle/trackers.py): round once, here.
    p.det_thresh = (float)cfg->conf_thresh;                                                   // basetrack.py:354
    p.low_thresh = (float)((cfg->conf_thresh - 0.3) > 0.15 ? (cfg->conf_thresh - 0.3) : 0.15);  // bytetrack.py:15
    p.new_thresh = (float)(cfg->conf_thresh + 0.1);                                           // bytetrack.py:175
    if (cfg->kind == B2T_SORT) { p.t1 = cfg->iou_thresh; p.t2 = 0.0; p.t3 = cfg->iou_thresh + 0.1; }   // basetrack.py:414,438
    else { p.t1 = 0.9; p.t2 = 0.5; p.t3 = 0.7; }                                              // bytetrack.py:118,137,160 ; c_biou_tracker.py:263,284,303
    p.t_dup = 0.15;                                                                           // basetrack.py:565
    p.max_time_lost = (int)(cfg->frame_rate / 30.0 * cfg->track_buffer);                      // basetrack.py:355-356
    p.use_gmc = cbiou ? 0 : cfg->use_gmc; p.predict_only = 0;
    if (cbiou) {
        t->smem = cbiou_smem_bytes(cfg->cap, cfg->dmax, t->st.esm);
        auto k = cbiou_step_kernel<double>;
        if (B2T_SET_SMEM(k, t->smem) != 0) { delete t; return fail(B2T_ECUDA, "cannot raise dynamic shared memory"); }
        *out = t;
        return b2t_tracker_reset(t, stream);
    }
    t->smem = cfg->dtype == B2T_F64 ? StepSmem<double>::bytes(cfg->cap, cfg->dmax, t->st.esm) : StepSmem<float>::bytes(cfg->cap, cfg->dmax, t->st.esm);
    if (cfg->dtype == B2T_F64) { auto k = track_step_kernel<double>; if (B2T_SET_SMEM(k, t->smem) != 0) { delete t; return fail(B2T_ECUDA, "cannot raise dynamic shared memory"); } }
    else { auto k = track_step_kernel<float>; if (B2T_SET_SMEM(k, t->smem) != 0) { delete t; return fail(B2T_ECUDA, "cannot raise dynamic shared memory"); } }
    *out = t;
    return b2t_tracker_reset(t, stream);
}

extern "C" void b2t_tracker_destroy(b2t_tracker* t) { delete t; }
extern "C" int b2t_tracker_out_cols(void) { return OUT_COLS; }
extern "C" int b2t_tracker_stat_words(void) { return STAT_WORDS; }

extern "C" int b2t_tracker_step(b2t_tracker* t, const float* dets, const int* det_count, const double* warps,
                                const int* id_base, double* out, int out_rows, int* stat, int predict_only, void* stream) {
    if (!t || !out || !stat || out_rows < 1) return fail(B2T_EINVAL, "b2t_tracker_step: bad arguments");
    if (!predict_only && (!dets || !det_count)) return fail(B2T_EINVAL, "b2t_tracker_step: dets / det_count are NULL");
    if (predict_only && t->cfg.kind == B2T_CBIOU)
        return fail(B2T_EINVAL, "b2t_tracker_step: predict_only is not defined for B2T_CBIOU (the reference's update_without_detection "
                                "predicts with a Kalman filter C-BIoU does not have)");
    StepParams p = t->prm;
    p.predict_only = predict_only ? 1 : 0;
    cudaStream_t s = (cudaStream_t)stream;
    if (t->cfg.kind == B2T_CBIOU) {
        auto k = cbiou_step_kernel<double>;
        B2T_LAUNCH(k, t->cfg.n_seq, 512, t->smem, s, t->st, p, dets, det_count, id_base, out, out_rows, stat);
    } else if (t->cfg.dtype == B2T_F64) {
        auto k = track_step_kernel<double>;
        B2T_LAUNCH(k, t->cfg.n_seq, 512, t->smem, s, t->st, p, dets, det_count, warps, id_base, out, out_rows, stat);
    } else {
        auto k = track_step_kernel<float>;
        B2T_LAUNCH(k, t->cfg.n_seq, 512, t->smem, s, t->st, p, dets, det_count, warps, id_base, out, out_rows, stat);
    }
    return check_launch("track_step");
}

extern "C" int b2t_tracker_step_host(b2t_tracker* t, const float* dets_host, const int* det_count_host,
                                     const double* warps_host, const int* id_base_host, double* out_host, int out_rows,
                                     int* stat_host, int predict_only, void* stream) {
    if (!t || !out_host || !stat_host) return fail(B2T_EINVAL, "b2t_tracker_step_host: bad arguments");
    if (predict_only && t->cfg.kind == B2T_CBIOU)
        return fail(B2T_EINVAL, "b2t_tracker_step_host: predict_only is not defined for B2T_CBIOU (the reference's update_without_detection "
                                "predicts with a Kalman filter C-BIoU does not have)");
    if (out_rows < 1 || (size_t)out_rows > t->out_rows_cap) return fail(B2T_EINVAL, "b2t_tracker_step_host: out_rows must be in [1, cap]");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t S = t->cfg.n_seq;
    if (!predict_only) {
        if (!dets_host || !det_count_host) return fail(B2T_EINVAL, "b2t_tracker_step_host: dets / det_count are NULL");
        cudaMemcpyAsync(t->d_dets, dets_host, sizeof(float) * S * t->cfg.dmax * 6, cudaMemcpyHostToDevice, s);
        cudaMemcpyAsync(t->d_count, det_count_host, sizeof(int) * S, cudaMemcpyHostToDevice, s);
    }
    if (warps_host) cudaMemcpyAsync(t->d_warps, warps_host, sizeof(double) * S * 6, cudaMemcpyHostToDevice, s);
    if (id_base_host) cudaMemcpyAsync(t->d_idbase, id_base_host, sizeof(int) * S, cudaMemcpyHostToDevice, s);
    int rc = b2t_tracker_step(t, t->d_dets, t->d_count, warps_host ? t->d_warps : nullptr, id_base_host ? t->d_idbase : nullptr,
                              t->d_out, out_rows, t->d_stat, predict_only, stream);
    if (rc) return rc;
    cudaMemcpyAsync(out_host, t->d_out, sizeof(double) * S * out_rows * OUT_COLS, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(stat_host, t->d_stat, sizeof(int) * S * STAT_WORDS, cudaMemcpyDeviceToHost, s);
    if (cudaStreamSynchronize(s) != cudaSuccess) return fail(B2T_ECUDA, "b2t_tracker_step_host: %s", cudaGetErrorString(cudaGetLastError()));
    for (size_t q = 0; q < S; ++q)
        if (stat_host[q * STAT_WORDS + STAT_ERR]) return fail(B2T_ECAPACITY, "b2t_tracker_step_host: capacity exceeded (cap / dmax / ecap), see stat[STAT_ERR]");
    return B2T_OK;
}

extern "C" int b2t_tracker_list_cols(void) { return LIST_COLS; }

extern "C" int b2t_tracker_read_list(b2t_tracker* t, int seq, int which, double* rows_host, int max_rows, int* n_host, void* stream) {
    if (!t || seq < 0 || seq >= t->cfg.n_seq || (which != 0 && which != 1) || !rows_host || !n_host || max_rows < 0)
        return fail(B2T_EINVAL, "b2t_tracker_read_list: bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    if (t->cfg.dtype == B2T_F64) { auto k = read_list_kernel<double>; B2T_LAUNCH(k, 1, 256, 0, s, t->st, t->cfg.kind, t->cfg.fmt, seq, which, t->d_list); }
    else { auto k = read_list_kernel<float>; B2T_LAUNCH(k, 1, 256, 0, s, t->st, t->cfg.kind, t->cfg.fmt, seq, which, t->d_list); }
    int rc = check_launch("read_list");
    if (rc) return rc;
    double nd = 0;
    cudaMemcpyAsync(&nd, t->d_list + (size_t)t->cfg.cap * LIST_COLS, sizeof nd, cudaMemcpyDeviceToHost, s);
    if (cudaStreamSynchronize(s) != cudaSuccess) return fail(B2T_ECUDA, "b2t_tracker_read_list: sync failed");
    int n = (int)nd;
    *n_host = n;
    if (n > max_rows) n = max_rows;
    if (n > 0) {
        cudaMemcpyAsync(rows_host, t->d_list, (size_t)n * LIST_COLS * sizeof(double), cudaMemcpyDeviceToHost, s);
        if (cudaStreamSynchronize(s) != cudaSuccess) return fail(B2T_ECUDA, "b2t_tracker_read_list: sync failed");
    }
    return B2T_OK;
}

extern "C" int b2t_tracker_read_slot(b2t_tracker* t, int seq, int slot, double* mean_host, double* cov_host, void* stream) {
    if (!t || seq < 0 || seq >= t->cfg.n_seq || slot < 0 || slot >= t->cfg.cap || !mean_host || !cov_host)
        return fail(B2T_EINVAL, "b2t_tracker_read_slot: bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    if (t->cfg.dtype == B2T_F64) { auto k = read_slot_kernel<double>; B2T_LAUNCH(k, 1, 64, 0, s, t->st, seq, slot, t->d_slot); }
    else { auto k = read_slot_kernel<float>; B2T_LAUNCH(k, 1, 64, 0, s, t->st, seq, slot, t->d_slot); }
    int rc = check_launch("read_slot");
    if (rc) return rc;
    double tmp[72];
    cudaMemcpyAsync(tmp, t->d_slot, sizeof tmp, cudaMemcpyDeviceToHost, s);
    if (cudaStreamSynchronize(s) != cudaSuccess) return fail(B2T_ECUDA, "b2t_tracker_read_slot: sync failed");
    memcpy(mean_host, tmp, 8 * sizeof(double));
    memcpy(cov_host, tmp + 8, 64 * sizeof(double));
    return B2T_OK;
}
