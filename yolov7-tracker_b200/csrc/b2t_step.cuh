// b2t_step.cuh -- the whole per-frame tracker update as ONE kernel, one CTA per video sequence.
//
// Replaces, for every sequence of the batch in a single launch,
//   BaseTracker.update   tracker/basetrack.py:368-487   (kind 0, SORT)
//   ByteTrack.update     tracker/bytetrack.py:41-204    (kind 1)
//   BoTSORT.update       tracker/botsort.py:313-493     (kind 2, + multi_gmc :250-269)
// including STrack.activate / update / re_activate / multi_predict (basetrack.py:222-339) and
// joint_stracks / sub_stracks / remove_duplicate_stracks (:540-576).  oracle/trackers.py is the
// CPU statement of the same machine; the quirk numbers (q3..q13) refer to SURVEY.md section 8a.
//
// HBM layout (per sequence s, slot-indexed SoA; T = double or float):
//   mean [S][cap][8] T, cov [S][cap][64] T          Kalman state, one 576-B (fp64) record per slot
//   tid/state/activated/tracklet_len/start_frame/frame_id/flags/removed_at [S][cap] int32
//   cls/score [S][cap] float32
//   tracked/lost/freelist [S][cap] int32            ordered slot lists (order defines row order, q13)
//   ctrl [S][16] int32                              frame, next_id, list lengths, error
//   e_col [S][ecap] int32, e_cost [S][ecap] T       CSR edges of the current association
// Everything else (boxes, lists, assignment state) lives in shared memory for the frame.
#pragma once
#include "b2t_prims.cuh"
#include "b2t_kalman.cuh"
#include "b2t_iou.cuh"
#include "b2t_lap.cuh"

namespace b2t {

enum { KIND_SORT = 0, KIND_BYTETRACK = 1, KIND_BOTSORT = 2 };
enum { ST_NEW = 0, ST_TRACKED = 1, ST_LOST = 2, ST_REMOVED = 3 };
enum { CTRL_FRAME = 0, CTRL_NEXT_ID = 1, CTRL_NTRACKED = 2, CTRL_NLOST = 3, CTRL_NFREE = 4, CTRL_ERR = 5 };
enum { STAT_NOUT = 0, STAT_NEXT_ID = 1, STAT_NTRACKED = 2, STAT_NLOST = 3, STAT_ERR = 4, STAT_FRAME = 5,
       STAT_NPOOL = 6, STAT_NBIRTH = 7, STAT_NHI = 8, STAT_NLO = 9, STAT_NEDGE = 10, STAT_NMATCH0 = 11,
       STAT_PHASE0 = 16,   // [16..32): SM cycles spent per phase (thread 0's clock64 deltas)
       STAT_SUB0 = 32,     // [32..64): sub-phase cycle stamps of association 1 (CSR build, LAP)
       STAT_WORDS = 64 };
enum { ERR_SLOTS = 1, ERR_EDGES = 2, ERR_DETS = 4, ERR_OUT = 8 };    // ERR_OUT: more confirmed tracks than output rows (rows were dropped)
enum { OUT_COLS = 8 };   // id, x, y, w, h, cls, score, slot
enum { NBINS = 64 };

struct TrackState {
    int n_seq, cap, dmax, ecap, esm;
    void* mean; void* cov;
    int *tid, *state, *activated, *tracklet_len, *start_frame, *frame_id, *flags, *removed_at;
    float *cls, *score;
    int *tracked, *lost, *freelist, *ctrl;
    int *e_col, *e_row; void* e_cost;
};

struct StepParams {
    int kind, fmt;
    float det_thresh, low_thresh, new_thresh;   // float32 comparisons, as NumPy 2 does them (oracle/trackers.py)
    double t1, t2, t3, t_dup;                   // association thresholds
    int max_time_lost;
    int use_gmc;
    int predict_only;                           // update_without_detection (basetrack.py:489-537)
};

template <class T> struct StepSmem {
    T *rowbox, *colbox, *detbox;
    int *hi, *lo, *pool, *unconf, *ut, *udets0, *lost_now, *births, *refind, *ntr, *nlo, *rcnt, *rstart;
    unsigned char *pstate, *dupa, *dupb, *used;
    int* misc;   // 64 ints
    int *perm, *bins;          // columns sorted by x1 bin; bins[0..NB] = start of each bin
    T* fmisc;                  // 8 values: column x-range, bin scale, max column width
    int *se_col, *se_row; T* se_cost; int esm;   // shared-memory mirror of the CSR edges (first esm entries)
    int box_bytes;             // rowbox + colbox: idle between build_csr and the next association -> second edge window (associate())
    LapWork<T> lap;
    template <class A> B2T_DEV void carve(A& a, int cap, int dmax, int esm_) {
        const int mx = cap > dmax ? cap : dmax;
        rowbox = a.template take<T>(4 * cap); colbox = a.template take<T>(4 * mx); detbox = a.template take<T>(4 * dmax);
        box_bytes = (int)(reinterpret_cast<unsigned char*>(colbox + 4 * mx) - reinterpret_cast<unsigned char*>(rowbox));
        hi = a.template take<int>(dmax); lo = a.template take<int>(dmax); pool = a.template take<int>(cap);
        unconf = a.template take<int>(cap); ut = a.template take<int>(cap); udets0 = a.template take<int>(dmax);
        lost_now = a.template take<int>(cap); births = a.template take<int>(dmax); refind = a.template take<int>(cap);
        ntr = a.template take<int>(cap); nlo = a.template take<int>(cap); rcnt = a.template take<int>(cap + 1);
        rstart = a.template take<int>(cap + 1);
        pstate = a.template take<unsigned char>(cap); dupa = a.template take<unsigned char>(cap);
        dupb = a.template take<unsigned char>(cap); used = a.template take<unsigned char>(cap);
        misc = a.template take<int>(64);
        perm = a.template take<int>(mx); bins = a.template take<int>(NBINS + 2); fmisc = a.template take<T>(8);
        lap.carve(a, cap, mx);
        esm = esm_;
        se_col = a.template take<int>(esm_); se_row = a.template take<int>(esm_); se_cost = a.template take<T>(esm_);
    }
    static size_t bytes(int cap, int dmax, int esm_) {
        ArenaSize a;
        const int mx = cap > dmax ? cap : dmax;
        a.take<T>(4 * cap); a.take<T>(4 * mx); a.take<T>(4 * dmax);
        a.take<int>(dmax); a.take<int>(dmax); a.take<int>(cap);
        a.take<int>(cap); a.take<int>(cap); a.take<int>(dmax);
        a.take<int>(cap); a.take<int>(dmax); a.take<int>(cap);
        a.take<int>(cap); a.take<int>(cap); a.take<int>(cap + 1); a.take<int>(cap + 1);
        a.take<unsigned char>(cap); a.take<unsigned char>(cap); a.take<unsigned char>(cap); a.take<unsigned char>(cap);
        a.take<int>(64);
        a.take<int>(mx); a.take<int>(NBINS + 2); a.take<T>(8);
        LapWork<T>::size(a, cap, mx);
        a.take<int>(esm_); a.take<int>(esm_); a.take<T>(esm_);
        return a.off + 16;
    }
    // largest shared-memory edge mirror that still fits next to everything else
    static int fit_esm(int cap, int dmax, int ecap, size_t limit) {
        const size_t base = bytes(cap, dmax, 0) + 64;
        if (base >= limit) return 0;
        size_t e = (limit - base) / (2 * sizeof(int) + sizeof(T));
        if (e > (size_t)ecap) e = (size_t)ecap;
        return (int)(e & ~size_t(3));
    }
};

#if defined(B2T_HOSTSIM)
B2T_DEV long long phase_clock() { return 0; }
#else
B2T_DEV long long phase_clock() { return clock64(); }
#endif
// sub-phase stamp: dbg (thread 0, may be null) receives cycles since the previous stamp
#define B2T_SUB(idx) do { if (dbg && threadIdx.x == 0) { const long long n_ = phase_clock(); dbg[idx] = (int)(n_ - *dbgt); *dbgt = n_; } } while (0)

// Per-sequence view of the global state.
template <class T> struct SeqView {
    T *mean, *cov, *e_cost;
    int *tid, *state, *activated, *tracklet_len, *start_frame, *frame_id, *flags, *removed_at;
    float *cls, *score;
    int *tracked, *lost, *freelist, *ctrl, *e_col, *e_row;
    int cap, ecap;
    B2T_DEV SeqView(const TrackState& st, int s) {
        const size_t c = (size_t)st.cap, o = (size_t)s * c;
        cap = st.cap; ecap = st.ecap;
        mean = (T*)st.mean + o * 8; cov = (T*)st.cov + o * 64;
        tid = st.tid + o; state = st.state + o; activated = st.activated + o; tracklet_len = st.tracklet_len + o;
        start_frame = st.start_frame + o; frame_id = st.frame_id + o; flags = st.flags + o; removed_at = st.removed_at + o;
        cls = st.cls + o; score = st.score + o;
        tracked = st.tracked + o; lost = st.lost + o; freelist = st.freelist + o;
        ctrl = st.ctrl + (size_t)s * 16;
        e_col = st.e_col + (size_t)s * st.ecap; e_row = st.e_row + (size_t)s * st.ecap; e_cost = (T*)st.e_cost + (size_t)s * st.ecap;
    }
};

// boxes of tracks listed in slots[0..n) -> box[k][0..4) (tlbr)
template <class T> B2T_DEV void fill_track_boxes(const SeqView<T>& v, int fmt, const int* slots, int n, T* box) {
    for (int k = (int)threadIdx.x; k < n; k += (int)blockDim.x) {
        const int s = slots[k];
        mean_to_tlbr<T>(fmt, v.mean + (size_t)s * 8, (v.flags[s] & 1) != 0, box + 4 * k);
    }
}

// Sparse cost rows: for every row box, the columns with (1 - IoU) < thresh, as CSR.
//   0. (m > 64 only) columns are counting-sorted by the x1 of their box into NBINS bins over the
//      column x-range (stable, one warp, __match_any); a row then only visits the bins whose x1 can
//      overlap it: x1 in [a.x1 - 2 - max_col_width, a.x2 + 2] (necessary for iw > 0, +1 convention);
//   1. one THREAD per row counts its candidates = boxes overlapping under the +1 convention (exact
//      compare, no division); an exclusive scan lays the rows out contiguously and deterministically;
//      the same threads then list their candidates' columns;
//   2. one thread per candidate pair evaluates the IoU (the fp64 division is ~60 SASS instructions):
//      exactly once per overlapping pair, all lanes busy.  Pairs at or above the threshold become
//      holes (col = -1) that every consumer skips;
//   3. rows whose range ends below esm live in shared memory, the others in the sequence's global
//      edge workspace (same indices) -- LapCsr::cols/costs picks per row.
// Requires m <= 1024.  Returns false (uniformly) on edge-workspace overflow.
template <class T>
B2T_DEVNI bool build_csr(SeqView<T>& v, StepSmem<T>& sm, int n, int m, T thresh, int* dbg = nullptr, long long* dbgt = nullptr) {
    const int tid = (int)threadIdx.x, nthr = (int)blockDim.x, lane = lane_id();
    int* misc = sm.misc;
    const T* colbox = sm.colbox;
    const bool sorted = m > 64;
    T xmin = (T)0, scale = (T)0, maxw = (T)0;
    if (tid == 0) { misc[50] = 0; misc[51] = 0; }
    if (sorted) {
        // ---- column statistics: min / max x1, max width
        T lo = (T)1e30, hi = (T)-1e30, mw = (T)0;
        for (int j = tid; j < m; j += nthr) {
            const T x1 = colbox[4 * j], wdt = colbox[4 * j + 2] - x1;
            lo = t_min(lo, x1); hi = t_max(hi, x1); mw = t_max(mw, wdt);
        }
        for (int o = 16; o; o >>= 1) {
            lo = t_min(lo, shfl_xor(lo, o)); hi = t_max(hi, shfl_xor(hi, o)); mw = t_max(mw, shfl_xor(mw, o));
        }
        for (int b = tid; b < NBINS + 2; b += nthr) sm.bins[b] = 0;
        if (lane == 0) { sm.lap.u[warp_id()] = lo; sm.lap.v[warp_id()] = hi; sm.lap.dist[warp_id()] = mw; }
        __syncthreads();
        if (tid < 32) {
            const bool on = tid < num_warps();
            T a = on ? sm.lap.u[tid] : (T)1e30, b = on ? sm.lap.v[tid] : (T)-1e30, c = on ? sm.lap.dist[tid] : (T)0;
            for (int o = 16; o; o >>= 1) { a = t_min(a, shfl_xor(a, o)); b = t_max(b, shfl_xor(b, o)); c = t_max(c, shfl_xor(c, o)); }
            if (tid == 0) {
                sm.fmisc[0] = a;
                sm.fmisc[1] = (b > a) ? (T)NBINS / ((b - a) * (T)1.0001 + (T)1e-3) : (T)0;
                sm.fmisc[2] = c;
            }
        }
        __syncthreads();
        xmin = sm.fmisc[0]; scale = sm.fmisc[1]; maxw = sm.fmisc[2];
    }
    B2T_SUB(0);
    auto bin_of = [&](T x) { T f = (x - xmin) * scale; int b = f > (T)0 ? (f < (T)(NBINS - 1) ? (int)f : NBINS - 1) : 0; return b; };
    if (sorted) {
        for (int j = tid; j < m; j += nthr) atomicAdd(&sm.bins[bin_of(colbox[4 * j])], 1);
        __syncthreads();
        if (warp_id() == 0) {
            // exclusive scan of the NBINS counts (2 per lane), then the stable scatter
            int c0 = sm.bins[2 * lane], c1 = sm.bins[2 * lane + 1];
            int sum = c0 + c1, inc = sum;
            for (int d = 1; d < 32; d <<= 1) { int t = shfl_up(inc, d); if (lane >= d) inc += t; }
            const int ex = inc - sum;
            __syncwarp();
            sm.bins[2 * lane] = ex; sm.bins[2 * lane + 1] = ex + c0;
            if (lane == 31) sm.bins[NBINS] = inc;
            sm.lap.cur[2 * lane] = ex; sm.lap.cur[2 * lane + 1] = ex + c0;      // per-bin cursor
            __syncwarp();
            for (int j0 = 0; j0 < m; j0 += 32) {
                const int j = j0 + lane;
                const int b = j < m ? bin_of(colbox[4 * j]) : -1;
                const unsigned mm = __match_any_sync(B2T_FULL, b);
                if (b >= 0) sm.perm[sm.lap.cur[b] + __popc(mm & lanemask_lt())] = j;
                __syncwarp();
                if (b >= 0 && (mm & lanemask_lt()) == 0) sm.lap.cur[b] += __popc(mm);
                __syncwarp();
            }
        }
    }
    __syncthreads();
    B2T_SUB(1);
    auto overlaps = [&](const T* a, const T* b) {
        return (t_min(a[2], b[2]) - t_max(a[0], b[0]) + (T)1 > (T)0) && (t_min(a[3], b[3]) - t_max(a[1], b[1]) + (T)1 > (T)0);
    };
    // ---- stage 1a: candidate count per row.  8 lanes per row (4 rows per warp): the lanes stride over
    // the row's candidate range, so a row costs ~range/8 dependent steps instead of range.
    const int sub = lane & 7, grp = lane >> 3;
    const unsigned gmask = 0xffu << (grp * 8);
    for (int base = warp_id() * 4; base < n; base += num_warps() * 4) {
        const int i = base + grp;
        const bool on = i < n;
        const T* a = sm.rowbox + 4 * (on ? i : 0);
        int k0 = 0, k1 = on ? m : 0;
        if (sorted && on) { k0 = sm.bins[bin_of(a[0] - (T)2 - maxw)]; k1 = sm.bins[bin_of(a[2] + (T)2) + 1]; }
        int cnt = 0;
        for (int k = k0 + sub; __any_sync(B2T_FULL, k < k1); k += 8) {
            const bool f = (k < k1) && overlaps(a, colbox + 4 * (sorted ? sm.perm[k] : k));
            cnt += __popc(__ballot_sync(B2T_FULL, f) & gmask);
        }
        if (on && sub == 0) { sm.rcnt[i] = cnt; sm.rstart[i] = cnt; }
    }
    if (tid == 0) sm.rstart[n] = 0;
    __syncthreads();
    B2T_SUB(2);
    const int total = block_exscan(sm.rstart, n + 1, sm.lap.scratch);
    B2T_SUB(3);
    const bool fits = total <= v.ecap;
    if (tid == 0) { misc[50] = total; misc[51] = fits ? 0 : 1; }
    // ---- stage 1b: list the candidates (same traversal, ordered by candidate position)
    if (fits) {
        for (int base = warp_id() * 4; base < n; base += num_warps() * 4) {
            const int i = base + grp;
            const bool on = i < n;
            const T* a = sm.rowbox + 4 * (on ? i : 0);
            int k0 = 0, k1 = on ? m : 0;
            if (sorted && on) { k0 = sm.bins[bin_of(a[0] - (T)2 - maxw)]; k1 = sm.bins[bin_of(a[2] + (T)2) + 1]; }
            const int cnt = on ? sm.rcnt[i] : 0;
            int pos = on ? sm.rstart[i] : 0;
            const bool to_smem = pos + cnt <= sm.esm;
            int* ocol = to_smem ? sm.se_col : v.e_col;
            int* orow = to_smem ? sm.se_row : v.e_row;
            for (int k = k0 + sub; __any_sync(B2T_FULL, k < k1); k += 8) {
                const int j = (k < k1) ? (sorted ? sm.perm[k] : k) : 0;
                const bool f = (k < k1) && overlaps(a, colbox + 4 * j);
                const unsigned bal = __ballot_sync(B2T_FULL, f) & gmask;
                if (f) { const int q = pos + __popc(bal & lanemask_lt()); ocol[q] = j; orow[q] = i; }
                pos += __popc(bal);
            }
        }
    } else {
        for (int i = tid; i < n; i += nthr) sm.rcnt[i] = 0;
    }
    __syncthreads();
    B2T_SUB(4);
    // ---- stage 2: one thread per candidate pair
    const int nE = fits ? total : 0;
    for (int e = tid; e < nE; e += nthr) {
        // which storage holds entry e?  rows never straddle: a row is in shared memory iff it ends below esm
        int* pc = sm.se_col; T* pw = sm.se_cost;
        int i = e < sm.esm ? sm.se_row[e] : -1;
        if (!(i >= 0 && i < n && sm.rstart[i] <= e && e < sm.rstart[i] + sm.rcnt[i] && sm.rstart[i] + sm.rcnt[i] <= sm.esm)) {
            pc = v.e_col; pw = v.e_cost; i = v.e_row[e];
        }
        const int j = pc[e];
        const T cost = (T)1 - iou_plus1<T>(sm.rowbox + 4 * i, colbox + 4 * j);
        if (cost < thresh) pw[e] = cost; else pc[e] = -1;
    }
    __syncthreads();
    B2T_SUB(5);
    return fits;
}

template <class T> struct StepCtx {
    SeqView<T> v;
    StepSmem<T> sm;
    StepParams p;
    int f;          // current frame id
    B2T_DEV StepCtx(const TrackState& st, int s, const StepParams& prm) : v(st, s), p(prm), f(0) {}
};

// thresholded assignment rows x cols; result in sm.lap.x / sm.lap.y.  tsplit (thread 0 only,
// may be null) receives the cycle count at the CSR / LAP boundary for the phase statistics.
template <class T> B2T_DEV LapCsr<T> step_csr(StepCtx<T>& c, int w2_base = 0, int w2_end = 0) {
    LapCsr<T> g;
    if (w2_end > w2_base) {
        const int cap2 = c.sm.box_bytes / (int)(sizeof(T) + 8);
        g.w2_cost = c.sm.rowbox; g.w2_col = reinterpret_cast<const int*>(c.sm.rowbox + cap2); g.w2_row = g.w2_col + cap2;
        g.w2_base = w2_base; g.w2_end = w2_end;
    }
    g.row_start = c.sm.rstart; g.row_stride = 0; g.row_cnt = c.sm.rcnt;
    g.e_col = c.v.e_col; g.e_cost = c.v.e_cost;
    g.s_col = c.sm.se_col; g.s_cost = c.sm.se_cost; g.s_cap = c.sm.esm;
    g.e_row = c.v.e_row; g.s_row = c.sm.se_row; g.n_entries = c.sm.misc[50] <= c.v.ecap ? c.sm.misc[50] : 0;
    return g;
}

template <class T> B2T_DEVNI void associate(StepCtx<T>& c, int n, int m, T thresh, int* err, long long* tsplit, int* dbg = nullptr) {
    StepSmem<T>& sm = c.sm;
    long long dt = phase_clock();
    const bool ok = build_csr<T>(c.v, sm, n, m, thresh, dbg, &dt);
    if (!ok && threadIdx.x == 0) *err |= ERR_EDGES;
    // The rows that did not fit the shared-memory edge mirror live in the global edge workspace.  rowbox / colbox are dead from
    // here to the next association (each one refills them): the first spilled rows are copied into that memory, so that the
    // solver's dependent loads stay on chip (measured under the pipeline's dense noise load: 7 000 edges, esm ~3 000 -- the
    // augmenting searches spent 1.5 M cycles per frame waiting for L2).
    int w2_base = 0, w2_end = 0;
    {
        const int tid = (int)threadIdx.x, nthr = (int)blockDim.x;
        const int total = ok ? sm.misc[50] : 0;
        if (total > sm.esm) {
            if (tid == 0) sm.misc[52] = 0x7fffffff;
            __syncthreads();
            for (int i = tid; i < n; i += nthr)
                if (sm.rcnt[i] > 0 && sm.rstart[i] + sm.rcnt[i] > sm.esm) atomicMin(&sm.misc[52], sm.rstart[i]);
            __syncthreads();
            const int cap2 = sm.box_bytes / (int)(sizeof(T) + 8);
            w2_base = sm.misc[52];
            if (w2_base < total && cap2 > 0) {
                w2_end = w2_base + cap2 < total ? w2_base + cap2 : total;
                T* wc = sm.rowbox; int* wj = reinterpret_cast<int*>(sm.rowbox + cap2); int* wi = wj + cap2;
                for (int e = w2_base + tid; e < w2_end; e += nthr) { wc[e - w2_base] = c.v.e_cost[e]; wj[e - w2_base] = c.v.e_col[e]; wi[e - w2_base] = c.v.e_row[e]; }
            } else w2_base = 0;
            __syncthreads();
        }
    }
    if (tsplit && threadIdx.x == 0) *tsplit = phase_clock();
    const LapCsr<T> g = step_csr<T>(c, w2_base, w2_end);
    lap_solve_cta<T>(n, m, g, thresh, sm.lap, dbg ? dbg + 8 : nullptr, &dt);
}

// Kalman correction of the tracks rows[k] (slots) matched to detections, 8 lanes per track.
//   rowdet[k]  : detection index (>= 0) or -1 to skip row k
//   rowmode[k] : 0 = STrack.update, 1 = STrack.re_activate
template <class T>
B2T_DEVNI void apply_matches(StepCtx<T>& c, const int* rows, int n, const float* dets, const int* rowdet,
                             const unsigned char* rowmode) {
    const int r = lane_id() & 7, grp = lane_id() >> 3;
    for (int base = warp_id() * 4; base < n; base += num_warps() * 4) {
        const int k = base + grp;
        int d = -1, slot = 0;
        if (k < n) { d = rowdet[k]; slot = rows[k]; }
        const bool on = d >= 0;
        KRow<T> kr;
        T z[4];
        bool f32 = false;
        float conf = -1.f;
        int md = 0;
        if (on) {
            kf_load<T>(kr, c.v.mean + (size_t)slot * 8, c.v.cov + (size_t)slot * 64, r);
            const float* dd = dets + 6 * d;
            det_to_meas<T>(c.p.fmt, dd[0], dd[1], dd[2], dd[3], z);
            f32 = (c.v.flags[slot] & 1) != 0;
            md = rowmode[k];
            if (c.p.fmt == FMT_NSA && md == 0) conf = dd[4];
        } else {
            kr.m = (T)1;
            for (int j = 0; j < 8; ++j) kr.p[j] = (j == r) ? (T)1 : (T)0;
            z[0] = z[1] = z[2] = z[3] = (T)0;
        }
        kf_update<T>(kr, r, c.p.fmt, z, f32, conf);
        if (on) {
            kf_store<T>(kr, c.v.mean + (size_t)slot * 8, c.v.cov + (size_t)slot * 64, r);
            if (r == 0) {
                c.v.flags[slot] &= ~1;
                c.v.frame_id[slot] = c.f;
                c.v.tracklet_len[slot] = md == 0 ? c.v.tracklet_len[slot] + 1 : 0;
                c.v.score[slot] = dets[6 * d + 4];
                c.v.state[slot] = ST_TRACKED;
                c.v.activated[slot] = 1;
            }
        }
    }
    __syncthreads();
}

#define B2T_PHASE(idx) do { if (tid == 0) { const long long now_ = phase_clock(); stat[STAT_PHASE0 + (idx)] = (int)(now_ - tprev); tprev = now_; } } while (0)

struct FrameLists { int nt, nl, nout, nfree; };

// P9-P11 of a frame, shared by every kind: list algebra (bytetrack.py:186-193), remove_duplicate_stracks (basetrack.py:563-576),
// the output rows of the activated tracks and the free list.  box(slot, tlbr, out[4]) writes a track's box as tlbr (duplicate
// test) or tlwh (output rows): the Kalman kinds read it from the mean, C-BIoU from its last matched detection.
// On entry the states of this frame are final, sm.births[0..nbirth) / sm.refind[0..nref) / sm.lost_now[0..nlostnow) hold slots.
template <class T, class BoxFn>
B2T_DEV FrameLists finish_lists(StepCtx<T>& c, BoxFn box, int n_tracked0, int n_lost0, int nbirth, int nref, int nlostnow,
                                double* out, int out_rows, int* err, int* stat, long long& tprev) {
    StepSmem<T>& sm = c.sm;
    SeqView<T>& v = c.v;
    const StepParams& p = c.p;
    const int tid = (int)threadIdx.x, nthr = (int)blockDim.x;
    const int cap = v.cap;
    const int f = c.f;
    // ---- P9: list algebra (bytetrack.py:186-193)
    int nt1 = block_compact(n_tracked0, [&](int k) { return v.state[v.tracked[k]] == ST_TRACKED; }, sm.ut, sm.misc);
    for (int k = tid; k < nt1; k += nthr) sm.ntr[k] = v.tracked[sm.ut[k]];
    for (int k = tid; k < nbirth; k += nthr) sm.ntr[nt1 + k] = sm.births[k];
    for (int k = tid; k < nref; k += nthr) sm.ntr[nt1 + nbirth + k] = sm.refind[k];
    nt1 += nbirth + nref;
    if (nt1 > cap) { nt1 = cap; if (tid == 0) *err |= ERR_SLOTS; }
    // old lost entries that were not re-found and whose id was not in the removed list before this frame
    int nl1 = block_compact(n_lost0, [&](int k) { const int s = v.lost[k];
        return v.state[s] != ST_TRACKED && !(v.removed_at[s] != 0 && v.removed_at[s] < f); }, sm.ut, sm.misc);
    for (int k = tid; k < nl1; k += nthr) sm.nlo[k] = v.lost[sm.ut[k]];
    __syncthreads();
    const int nl_add = block_compact(nlostnow, [&](int k) { const int s = sm.lost_now[k];
        return !(v.removed_at[s] != 0 && v.removed_at[s] < f); }, sm.ut, sm.misc);
    for (int k = tid; k < nl_add; k += nthr) sm.nlo[nl1 + k] = sm.lost_now[sm.ut[k]];
    nl1 += nl_add;
    __syncthreads();

    B2T_PHASE(10);
    // ---- P10: remove_duplicate_stracks (basetrack.py:563-576)
    for (int k = tid; k < cap; k += nthr) { sm.dupa[k] = 0; sm.dupb[k] = 0; }
    for (int k = tid; k < nt1; k += nthr) box(sm.ntr[k], true, sm.rowbox + 4 * k);
    for (int k = tid; k < nl1; k += nthr) box(sm.nlo[k], true, sm.colbox + 4 * k);
    __syncthreads();
    if (nt1 > 0 && nl1 > 0) {
        const bool ok = build_csr<T>(v, sm, nt1, nl1, (T)p.t_dup);
        if (!ok && tid == 0) *err |= ERR_EDGES;
        const LapCsr<T> g = step_csr<T>(c);
        for (int i = warp_id(); i < nt1; i += num_warps()) {
            const int sa = sm.ntr[i];
            const int timep = v.frame_id[sa] - v.start_frame[sa];
            const int es = sm.rstart[i], ec = sm.rcnt[i];
            const int* ecol = g.cols(es, ec);
            for (int e = lane_id(); e < ec; e += 32) {
                const int q = ecol[e];
                if (q < 0) continue;
                const int sb = sm.nlo[q];
                const int timeq = v.frame_id[sb] - v.start_frame[sb];
                if (timep > timeq) sm.dupb[q] = 1; else sm.dupa[i] = 1;
            }
        }
        __syncthreads();
    }
    const int nt2 = block_compact(nt1, [&](int k) { return sm.dupa[k] == 0; }, sm.ut, sm.misc);
    for (int k = tid; k < nt2; k += nthr) v.tracked[k] = sm.ntr[sm.ut[k]];
    const int nl2 = block_compact(nl1, [&](int k) { return sm.dupb[k] == 0; }, sm.ut, sm.misc);
    for (int k = tid; k < nl2; k += nthr) v.lost[k] = sm.nlo[sm.ut[k]];
    for (int k = tid; k < cap; k += nthr) sm.used[k] = 0;
    __syncthreads();

    B2T_PHASE(11);
    // ---- P11: output rows (activated tracks, bytetrack.py:204) and the free list
    for (int k = tid; k < nt2; k += nthr) sm.used[v.tracked[k]] = 1;
    for (int k = tid; k < nl2; k += nthr) sm.used[v.lost[k]] = 1;
    __syncthreads();
    int nout = block_compact(nt2, [&](int k) { return v.activated[v.tracked[k]] != 0; }, sm.ut, sm.misc);
    if (nout > out_rows) { nout = out_rows; if (tid == 0) *err |= ERR_OUT; }
    for (int k = tid; k < nout; k += nthr) {
        const int s = v.tracked[sm.ut[k]];
        T b[4];
        box(s, false, b);
        double* o = out + (size_t)k * OUT_COLS;
        o[0] = (double)v.tid[s];
        o[1] = (double)b[0]; o[2] = (double)b[1]; o[3] = (double)b[2]; o[4] = (double)b[3];
        o[5] = (double)v.cls[s]; o[6] = (double)v.score[s]; o[7] = (double)s;
    }
    const int nfree2 = block_compact(cap, [&](int k) { return sm.used[k] == 0; }, v.freelist, sm.misc);
    B2T_PHASE(12);
    return FrameLists{nt2, nl2, nout, nfree2};
}

template <class T>
B2T_DEV void track_step_cta(const TrackState& st, const StepParams& prm, int seq, const float* dets_all,
                            const int* det_count, const double* warps, const int* id_base, double* out_all,
                            int out_rows, int* stat_all, unsigned char* smem_raw) {
    StepCtx<T> c(st, seq, prm);
    Arena arena(smem_raw);
    c.sm.carve(arena, st.cap, st.dmax, st.esm);
    StepSmem<T>& sm = c.sm;
    SeqView<T>& v = c.v;
    const StepParams& p = c.p;
    const int tid = (int)threadIdx.x, nthr = (int)blockDim.x;
    const int cap = st.cap;
    const float* dets = dets_all + (size_t)seq * st.dmax * 6;
    double* out = out_all + (size_t)seq * out_rows * OUT_COLS;
    int* stat = stat_all + (size_t)seq * STAT_WORDS;
    int* err = &sm.misc[48];
    long long tprev = phase_clock();

    if (tid == 0) {
        for (int q = 0; q < 48; ++q) stat[STAT_PHASE0 + q] = 0;
        *err = v.ctrl[CTRL_ERR];
        if (id_base) v.ctrl[CTRL_NEXT_ID] = id_base[seq];
        v.ctrl[CTRL_FRAME] += 1;
    }
    __syncthreads();
    c.f = v.ctrl[CTRL_FRAME];
    const int f = c.f;
    int nd = p.predict_only ? 0 : det_count[seq];
    if (nd > st.dmax) { nd = st.dmax; if (tid == 0) *err |= ERR_DETS; }
    const int n_tracked0 = v.ctrl[CTRL_NTRACKED], n_lost0 = v.ctrl[CTRL_NLOST];

    // ---- P0: detections -> boxes, high / low lists (bytetrack.py:69-74 ; basetrack.py:387)
    for (int i = tid; i < nd; i += nthr) {
        const float* d = dets + 6 * i;
        const float w = d[2] - d[0], h = d[3] - d[1];          // tlbr2tlwh, float32
        sm.detbox[4 * i + 0] = (T)d[0];
        sm.detbox[4 * i + 1] = (T)d[1];
        sm.detbox[4 * i + 2] = (T)(w + d[0]);                   // .tlbr: tlwh[2:] += tlwh[:2], float32
        sm.detbox[4 * i + 3] = (T)(h + d[1]);
    }
    int nhi, nlo;
    if (p.kind == KIND_SORT) {
        nhi = block_compact(nd, [&](int i) { return dets[6 * i + 4] > p.det_thresh; }, sm.hi, sm.misc);
        nlo = 0;
    } else {
        nhi = block_compact(nd, [&](int i) { return dets[6 * i + 4] >= p.det_thresh; }, sm.hi, sm.misc);
        nlo = block_compact(nd, [&](int i) { const float s = dets[6 * i + 4]; return !(s >= p.det_thresh) && s > p.low_thresh; },
                            sm.lo, sm.misc);
    }

    B2T_PHASE(0);
    // ---- P1: unconfirmed / confirmed split, pool = confirmed ++ lost (joint_stracks)
    const int nunc = block_compact(n_tracked0, [&](int k) { return v.activated[v.tracked[k]] == 0; }, sm.ut, sm.misc);
    for (int k = tid; k < nunc; k += nthr) sm.unconf[k] = v.tracked[sm.ut[k]];
    const int nconf = block_compact(n_tracked0, [&](int k) { return v.activated[v.tracked[k]] != 0; }, sm.ut, sm.misc);
    for (int k = tid; k < nconf; k += nthr) sm.pool[k] = v.tracked[sm.ut[k]];
    for (int k = tid; k < n_lost0; k += nthr) sm.pool[nconf + k] = v.lost[k];
    const int npool = nconf + n_lost0;
    if (tid == 0) sm.misc[49] = 1;
    __syncthreads();
    for (int k = tid; k < npool; k += nthr) {
        const int s = sm.pool[k];
        sm.pstate[k] = (unsigned char)v.state[s];
        if (!(v.flags[s] & 1)) sm.misc[49] = 0;
    }
    __syncthreads();
    const bool q_f32 = sm.misc[49] != 0;

    B2T_PHASE(1);
    // ---- P2: Kalman predict (+ camera-motion warp) for the pool, warp for the unconfirmed
    T warp6[6];
    const bool gmc = p.use_gmc && p.kind == KIND_BOTSORT && warps != nullptr && !p.predict_only;
    if (gmc) for (int q = 0; q < 6; ++q) warp6[q] = (T)warps[(size_t)seq * 6 + q];
    {
        const int r = lane_id() & 7, grp = lane_id() >> 3;
        for (int base = warp_id() * 4; base < npool; base += num_warps() * 4) {
            const int k = base + grp;
            const bool on = k < npool;
            const int slot = on ? sm.pool[k] : 0;
            KRow<T> kr;
            if (on) kf_load<T>(kr, v.mean + (size_t)slot * 8, v.cov + (size_t)slot * 64, r);
            else { kr.m = (T)0; for (int j = 0; j < 8; ++j) kr.p[j] = (T)0; }
            kf_predict<T>(kr, r, p.fmt, on && sm.pstate[k] != ST_TRACKED, q_f32);
            if (gmc) kf_gmc<T>(kr, r, warp6);
            if (on) {
                kf_store<T>(kr, v.mean + (size_t)slot * 8, v.cov + (size_t)slot * 64, r);
                if (r == 0) v.flags[slot] &= ~1;
            }
        }
        if (gmc) {
            for (int base = warp_id() * 4; base < nunc; base += num_warps() * 4) {
                const int k = base + grp;
                const bool on = k < nunc;
                const int slot = on ? sm.unconf[k] : 0;
                KRow<T> kr;
                if (on) kf_load<T>(kr, v.mean + (size_t)slot * 8, v.cov + (size_t)slot * 64, r);
                else { kr.m = (T)0; for (int j = 0; j < 8; ++j) kr.p[j] = (T)0; }
                kf_gmc<T>(kr, r, warp6);
                if (on) {
                    kf_store<T>(kr, v.mean + (size_t)slot * 8, v.cov + (size_t)slot * 64, r);
                    if (r == 0) v.flags[slot] &= ~1;
                }
            }
        }
    }
    __syncthreads();

    B2T_PHASE(2);
    int nref = 0, nlostnow = 0, nud0 = 0, nbirth = 0, nmatch0 = 0;
    if (!p.predict_only) {
        // ---- P3/P4: association 1, pool x high detections
        fill_track_boxes<T>(v, p.fmt, sm.pool, npool, sm.rowbox);
        for (int k = tid; k < nhi; k += nthr)
            for (int q = 0; q < 4; ++q) sm.colbox[4 * k + q] = sm.detbox[4 * sm.hi[k] + q];
        __syncthreads();
        B2T_PHASE(3);
        long long tsplit = tprev;
        associate<T>(c, npool, nhi, (T)p.t1, err, &tsplit, stat + STAT_SUB0);
        if (tid == 0) { stat[STAT_PHASE0 + 4] = (int)(tsplit - tprev); tprev = tsplit;
                        stat[12] = sm.lap.scratch[45]; stat[13] = sm.lap.scratch[41]; stat[14] = sm.lap.scratch[43]; stat[15] = sm.misc[50]; }
        B2T_PHASE(5);
        const int* x = sm.lap.x;
        const int* y = sm.lap.y;
        const bool sort = p.kind == KIND_SORT;
        // refind list (pre-update states), leftovers for the later stages
        nref = block_compact(npool, [&](int i) {
            return x[i] >= 0 && (sort ? sm.pstate[i] != ST_TRACKED : sm.pstate[i] == ST_LOST); }, sm.ntr, sm.misc);
        for (int k = tid; k < nref; k += nthr) sm.refind[k] = sm.pool[sm.ntr[k]];
        nud0 = block_compact(nhi, [&](int cidx) { return y[cidx] < 0; }, sm.ntr, sm.misc);
        for (int k = tid; k < nud0; k += nthr) sm.udets0[k] = sm.hi[sm.ntr[k]];
        int nut;
        if (sort)
            nut = block_compact(npool, [&](int i) { return x[i] < 0 && sm.pstate[i] == ST_TRACKED; }, sm.ut, sm.misc);
        else if (p.kind == KIND_BYTETRACK)
            nut = block_compact(npool, [&](int i) { return x[i] < 0 && sm.pstate[i] == ST_TRACKED; }, sm.ut, sm.misc);
        else
            nut = block_compact(npool, [&](int i) { return x[i] < 0; }, sm.ut, sm.misc);
        nmatch0 = npool - block_compact(npool, [&](int i) { return x[i] < 0; }, sm.ntr, sm.misc);
        for (int k = tid; k < npool; k += nthr) {
            const int xx = x[k], ps = sm.pstate[k];
            sm.ntr[k] = (xx >= 0 && (ps == ST_TRACKED || ps == ST_LOST || sort)) ? sm.hi[xx] : -1;
            sm.used[k] = ps == ST_TRACKED ? 0 : 1;
        }
        __syncthreads();
        apply_matches<T>(c, sm.pool, npool, dets, sm.ntr, sm.used);
        B2T_PHASE(6);
        if (sort) {
            // basetrack.py:429-433: unmatched Tracked rows become lost
            for (int k = tid; k < nut; k += nthr) { const int s = sm.pool[sm.ut[k]]; v.state[s] = ST_LOST; sm.lost_now[k] = s; }
            nlostnow = nut;
            __syncthreads();
        } else {
            // ---- P5: association 2, leftover tracks x low detections (thresh 0.5)
            for (int k = tid; k < nut; k += nthr) {
                sm.nlo[k] = sm.pool[sm.ut[k]];                                         // slots of u_tracks0
                sm.dupb[k] = sm.pstate[sm.ut[k]];                                      // their frame-start states
            }
            __syncthreads();
            fill_track_boxes<T>(v, p.fmt, sm.nlo, nut, sm.rowbox);
            for (int k = tid; k < nlo; k += nthr)
                for (int q = 0; q < 4; ++q) sm.colbox[4 * k + q] = sm.detbox[4 * sm.lo[k] + q];
            __syncthreads();
            associate<T>(c, nut, nlo, (T)p.t2, err, nullptr);
            const int nref2 = block_compact(nut, [&](int i) { return x[i] >= 0 && sm.dupb[i] == ST_LOST; }, sm.ntr, sm.misc);
            for (int k = tid; k < nref2; k += nthr) sm.refind[nref + k] = sm.nlo[sm.ntr[k]];
            const int nl = block_compact(nut, [&](int i) { return x[i] < 0; }, sm.ntr, sm.misc);
            // lost_now keeps only rows that were Tracked at frame start: the others are already in
            // the lost list and sub_stracks' id-dict would drop the second copy (q4).
            for (int k = tid; k < nl; k += nthr) { const int s = sm.nlo[sm.ntr[k]]; v.state[s] = ST_LOST; }
            nlostnow = block_compact(nl, [&](int k) { return sm.dupb[sm.ntr[k]] == ST_TRACKED; }, sm.ut, sm.misc);
            for (int k = tid; k < nlostnow; k += nthr) sm.lost_now[k] = sm.nlo[sm.ntr[sm.ut[k]]];
            __syncthreads();
            for (int k = tid; k < nut; k += nthr) {
                const int xx = x[k], ps = sm.dupb[k];
                sm.ntr[k] = (xx >= 0 && (ps == ST_TRACKED || ps == ST_LOST)) ? sm.lo[xx] : -1;
                sm.used[k] = ps == ST_TRACKED ? 0 : 1;
            }
            __syncthreads();
            apply_matches<T>(c, sm.nlo, nut, dets, sm.ntr, sm.used);
            nref += nref2;
        }

        B2T_PHASE(7);
        // ---- P6: association 3, unconfirmed x leftover high detections
        fill_track_boxes<T>(v, p.fmt, sm.unconf, nunc, sm.rowbox);
        for (int k = tid; k < nud0; k += nthr)
            for (int q = 0; q < 4; ++q) sm.colbox[4 * k + q] = sm.detbox[4 * sm.udets0[k] + q];
        __syncthreads();
        associate<T>(c, nunc, nud0, (T)p.t3, err, nullptr);
        for (int k = tid; k < nunc; k += nthr)
            if (x[k] < 0) { const int s = sm.unconf[k]; v.state[s] = ST_REMOVED; if (v.removed_at[s] == 0) v.removed_at[s] = f; }
        // births (q3: BoT-SORT walks every first-stage leftover, the others only third-stage leftovers)
        if (p.kind == KIND_BOTSORT)
            nbirth = block_compact(nud0, [&](int k) { return dets[6 * sm.udets0[k] + 4] > p.new_thresh; }, sm.ntr, sm.misc);
        else
            nbirth = block_compact(nud0, [&](int k) { return y[k] < 0 && dets[6 * sm.udets0[k] + 4] > p.new_thresh; },
                                   sm.ntr, sm.misc);
        for (int k = tid; k < nbirth; k += nthr) sm.births[k] = sm.udets0[sm.ntr[k]];      // det indices
        __syncthreads();
        for (int k = tid; k < nunc; k += nthr) { const int xx = x[k]; sm.ntr[k] = xx < 0 ? -1 : sm.udets0[xx]; sm.used[k] = 0; }
        __syncthreads();
        apply_matches<T>(c, sm.unconf, nunc, dets, sm.ntr, sm.used);

        B2T_PHASE(8);
        // ---- P7: births (STrack.activate, basetrack.py:222-245)
        const int nfree = v.ctrl[CTRL_NFREE];
        if (nbirth > nfree) { if (tid == 0) *err |= ERR_SLOTS; nbirth = nfree; }
        const int id0 = v.ctrl[CTRL_NEXT_ID];
        {
            const int r = lane_id() & 7, grp = lane_id() >> 3;
            for (int base = warp_id() * 4; base < nbirth; base += num_warps() * 4) {
                const int k = base + grp;
                if (k < nbirth) {
                    const int d = sm.births[k];
                    const int slot = v.freelist[k];
                    const float* dd = dets + 6 * d;
                    T z[4];
                    det_to_meas<T>(p.fmt, dd[0], dd[1], dd[2], dd[3], z);
                    KRow<T> kr;
                    kf_initiate<T>(kr, r, p.fmt, z);
                    kf_store<T>(kr, v.mean + (size_t)slot * 8, v.cov + (size_t)slot * 64, r);
                    if (r == 0) {
                        v.tid[slot] = id0 + 1 + k;
                        v.state[slot] = ST_TRACKED;
                        v.activated[slot] = (f == 1) ? 1 : 0;
                        v.tracklet_len[slot] = 0;
                        v.start_frame[slot] = f; v.frame_id[slot] = f;
                        v.flags[slot] = 1;
                        v.removed_at[slot] = 0;
                        v.cls[slot] = dd[5]; v.score[slot] = dd[4];
                    }
                }
            }
        }
        __syncthreads();
        for (int k = tid; k < nbirth; k += nthr) sm.births[k] = v.freelist[k];               // now slots
        if (tid == 0) v.ctrl[CTRL_NEXT_ID] = id0 + nbirth;
        // ---- P8: prune long-lost tracks (iterates the OLD lost list, bytetrack.py:180-183)
        for (int k = tid; k < n_lost0; k += nthr) {
            const int s = v.lost[k];
            if (f - v.frame_id[s] > p.max_time_lost) { v.state[s] = ST_REMOVED; if (v.removed_at[s] == 0) v.removed_at[s] = f; }
        }
        __syncthreads();
    }

    B2T_PHASE(9);
    auto kalman_box = [&](int s, bool tlbr, T* box) {
        if (tlbr) mean_to_tlbr<T>(p.fmt, v.mean + (size_t)s * 8, (v.flags[s] & 1) != 0, box);
        else mean_to_tlwh<T>(p.fmt, v.mean + (size_t)s * 8, (v.flags[s] & 1) != 0, box);
    };
    const FrameLists fl = finish_lists<T>(c, kalman_box, n_tracked0, n_lost0, nbirth, nref, nlostnow, out, out_rows, err, stat, tprev);
    if (tid == 0) {
        v.ctrl[CTRL_NTRACKED] = fl.nt; v.ctrl[CTRL_NLOST] = fl.nl; v.ctrl[CTRL_NFREE] = fl.nfree; v.ctrl[CTRL_ERR] = *err;
        stat[STAT_NOUT] = fl.nout; stat[STAT_NEXT_ID] = v.ctrl[CTRL_NEXT_ID]; stat[STAT_NTRACKED] = fl.nt; stat[STAT_NLOST] = fl.nl;
        stat[STAT_ERR] = *err; stat[STAT_FRAME] = f; stat[STAT_NPOOL] = npool; stat[STAT_NBIRTH] = nbirth;
        stat[STAT_NHI] = nhi; stat[STAT_NLO] = nlo; stat[STAT_NEDGE] = sm.misc[50]; stat[STAT_NMATCH0] = nmatch0;
    }
}

}  // namespace b2t
