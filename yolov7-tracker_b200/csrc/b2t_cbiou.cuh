// b2t_cbiou.cuh -- the C-BIoU tracker (C_BIoUTracker.update, tracker/c_biou_tracker.py:218-353) as ONE kernel, one CTA per
// video sequence.  Cascaded buffered IoU (Yang et al., "Hard to Track Objects with Irregular Motions and Similar Appearances?
// Make It Easier by Buffering the Matching Space", WACV 2023): no Kalman filter, three IoU associations on boxes enlarged by
// a buffer scale b (b1 = 0.3, b2 = 0.5), then the list algebra of ByteTrack (finish_lists, b2t_step.cuh).  fp64 only: the
// reference's IoU is float64 and its box arithmetic float32 (each operation rounded, --fmad=false).  oracle/cbiou.py is the CPU
// statement of the same machine.
//
// Slot record.  The Kalman kinds keep mean[8] + cov[64] doubles per slot; C-BIoU reuses those 72 doubles (r[0..8) = the mean
// array, r[8..72) = the cov array, b2t_tracker_read_slot returns them in this order):
//   r[0]        history length n (1..6)
//   r[1]        time_since_update
//   r[8..32)    history: n original tlwh boxes, oldest first (origin_bbox_buffer; trimmed when n > 5, before the append)
//   r[32..36)   motion_state1 (tlwh, buffer level b1)
//   r[36..40)   motion_state2 (tlwh, buffer level b2)
// Every box value is a float32 held in a double.
#pragma once
#include "b2t_step.cuh"

namespace b2t {

enum { KIND_CBIOU = 3 };
enum { CB_LEN = 0, CB_TSU = 1, CB_HIST = 0, CB_MS1 = 24, CB_MS2 = 28 };   // CB_LEN / CB_TSU index the mean part, the rest the cov part

// get_buffer_bbox (c_biou_tracker.py:48-62) in float32: max(0, [x - b w, y - b h, w + 2b w, h + 2b h]), nb = f32(-b), b2 = f32(2b)
B2T_DEV void cb_buffer(const float* t, float nb, float b2, float* o) {
    float r[4];
    r[0] = t[0] + nb * t[2]; r[1] = t[1] + nb * t[3]; r[2] = t[2] + b2 * t[2]; r[3] = t[3] + b2 * t[3];
    for (int q = 0; q < 4; ++q) o[q] = r[q] < 0.f ? 0.f : r[q];
}
B2T_DEV void cb_level1(const float* t, float* o) { cb_buffer(t, -0.3f, 0.6f, o); }
B2T_DEV void cb_level2(const float* t, float* o) { cb_buffer(t, -0.5f, 1.0f, o); }

// tlwh (float32 values) -> tlbr in float32 (tlwh2tlbr), widened
template <class T, class S> B2T_DEV void cb_tlbr(const S* tlwh, T* o) {
    const float x = (float)tlwh[0], y = (float)tlwh[1], w = (float)tlwh[2], h = (float)tlwh[3];
    o[0] = (T)x; o[1] = (T)y; o[2] = (T)(x + w); o[3] = (T)(y + h);
}

// detection -> float32 tlwh (tlbr2tlwh)
B2T_DEV void cb_det_tlwh(const float* d, float* t) { t[0] = d[0]; t[1] = d[1]; t[2] = d[2] - d[0]; t[3] = d[3] - d[1]; }

template <class T> B2T_DEV void cb_store4(T* dst, const float* s) { for (int q = 0; q < 4; ++q) dst[q] = (T)s[q]; }

// STrack.update (mode 0, :114-152) / re_activate (mode 1, :89-112) of the tracks rows[k] matched to detections rowdet[k]
// (-1 = skip), one thread per track.  re_activate keeps time_since_update: the next update extrapolates with it.
template <class T>
B2T_DEVNI void cb_apply(StepCtx<T>& c, const int* rows, int n, const float* dets, const int* rowdet, const unsigned char* rowmode) {
    for (int k = (int)threadIdx.x; k < n; k += (int)blockDim.x) {
        const int d = rowdet[k];
        if (d < 0) continue;
        const int s = rows[k], md = rowmode[k];
        T* rm = c.v.mean + (size_t)s * 8;
        T* rc = c.v.cov + (size_t)s * 64;
        float t[4];
        cb_det_tlwh(dets + 6 * d, t);
        int len = (int)rm[CB_LEN];
        if (len > 5) { for (int q = 0; q < 20; ++q) rc[CB_HIST + q] = rc[CB_HIST + 4 + q]; len = 5; }
        cb_store4(rc + CB_HIST + 4 * len, t);
        len += 1;
        rm[CB_LEN] = (T)len;
        const int tsu = (int)rm[CB_TSU];
        float src[4] = {t[0], t[1], t[2], t[3]};
        if (md == 0 && tsu != 0 && len >= 5) {
            // s = o_t + (tsu / n) (o_t - o_{t-n}), float32 with a float64 factor rounded once
            const float a = (float)((double)tsu / 5.0);
            for (int q = 0; q < 4; ++q) { const float o0 = (float)rc[CB_HIST + q]; src[q] = t[q] + a * (t[q] - o0); }
        }
        float b[4];
        cb_level1(src, b); cb_store4(rc + CB_MS1, b);
        cb_level2(src, b); cb_store4(rc + CB_MS2, b);
        if (md == 0) { rm[CB_TSU] = (T)0; c.v.tracklet_len[s] += 1; }
        else c.v.tracklet_len[s] = 0;
        c.v.frame_id[s] = c.f;
        c.v.score[s] = dets[6 * d + 4];
        c.v.state[s] = ST_TRACKED;
        c.v.activated[s] = 1;
    }
    __syncthreads();
}

// motion states (level 1: r[32..36), level 2: r[36..40)) of the tracks in slots[0..n) -> tlbr rows
template <class T> B2T_DEV void cb_fill_ms(const SeqView<T>& v, int off, const int* slots, int n, T* box) {
    for (int k = (int)threadIdx.x; k < n; k += (int)blockDim.x) cb_tlbr<T>(v.cov + (size_t)slots[k] * 64 + off, box + 4 * k);
}

template <class T>
B2T_DEV void cbiou_step_cta(const TrackState& st, const StepParams& prm, int seq, const float* dets_all, const int* det_count,
                            const int* id_base, double* out_all, int out_rows, int* stat_all, unsigned char* smem_raw) {
    StepCtx<T> c(st, seq, prm);
    Arena arena(smem_raw);
    c.sm.carve(arena, st.cap, st.dmax, st.esm);
    // buffered detection boxes (tlbr, float32 values): level 1 in buf[0..4 dmax), level 2 in buf[4 dmax..8 dmax) -- the storage of
    // sm.detbox, which only the Kalman kinds use
    static_assert(sizeof(T) == 2 * sizeof(float), "C-BIoU runs in fp64");
    float* buf1 = reinterpret_cast<float*>(c.sm.detbox);
    float* buf2 = buf1 + 4 * st.dmax;
    StepSmem<T>& sm = c.sm;
    SeqView<T>& v = c.v;
    const StepParams& p = c.p;
    const int tid = (int)threadIdx.x, nthr = (int)blockDim.x;
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
    int nd = det_count[seq];
    if (nd > st.dmax) { nd = st.dmax; if (tid == 0) *err |= ERR_DETS; }
    const int n_tracked0 = v.ctrl[CTRL_NTRACKED], n_lost0 = v.ctrl[CTRL_NLOST];

    // ---- P0: buffered boxes of every detection (the detection tracks' buffer_bbox1 / 2, :41-42), kept = score > det_thresh (:238)
    for (int i = tid; i < nd; i += nthr) {
        float t[4], b[4];
        cb_det_tlwh(dets + 6 * i, t);
        cb_level1(t, b);
        cb_tlbr<float>(b, buf1 + 4 * i);
        cb_level2(t, b);
        cb_tlbr<float>(b, buf2 + 4 * i);
    }
    const int nhi = block_compact(nd, [&](int i) { return dets[6 * i + 4] > p.det_thresh; }, sm.hi, sm.misc);

    B2T_PHASE(0);
    // ---- P1: unconfirmed / confirmed split, pool = confirmed ++ lost (:250-259)
    const int nunc = block_compact(n_tracked0, [&](int k) { return v.activated[v.tracked[k]] == 0; }, sm.ut, sm.misc);
    for (int k = tid; k < nunc; k += nthr) sm.unconf[k] = v.tracked[sm.ut[k]];
    const int nconf = block_compact(n_tracked0, [&](int k) { return v.activated[v.tracked[k]] != 0; }, sm.ut, sm.misc);
    for (int k = tid; k < nconf; k += nthr) sm.pool[k] = v.tracked[sm.ut[k]];
    for (int k = tid; k < n_lost0; k += nthr) sm.pool[nconf + k] = v.lost[k];
    const int npool = nconf + n_lost0;
    __syncthreads();
    for (int k = tid; k < npool; k += nthr) sm.pstate[k] = (unsigned char)v.state[sm.pool[k]];
    __syncthreads();

    B2T_PHASE(1);
    // ---- stage 1: pool motion_state1 x kept detections' level-1 buffers, threshold 0.9 (:261-275)
    cb_fill_ms<T>(v, CB_MS1, sm.pool, npool, sm.rowbox);
    for (int k = tid; k < nhi; k += nthr)
        for (int q = 0; q < 4; ++q) sm.colbox[4 * k + q] = (T)buf1[4 * sm.hi[k] + q];
    __syncthreads();
    B2T_PHASE(3);
    long long tsplit = tprev;
    associate<T>(c, npool, nhi, (T)p.t1, err, &tsplit, stat + STAT_SUB0);
    if (tid == 0) { stat[STAT_PHASE0 + 4] = (int)(tsplit - tprev); tprev = tsplit;
                    stat[12] = sm.lap.scratch[45]; stat[13] = sm.lap.scratch[41]; stat[14] = sm.lap.scratch[43]; stat[15] = sm.misc[50]; }
    B2T_PHASE(5);
    const int* x = sm.lap.x;
    const int* y = sm.lap.y;
    int nref = block_compact(npool, [&](int i) { return x[i] >= 0 && sm.pstate[i] == ST_LOST; }, sm.ntr, sm.misc);
    for (int k = tid; k < nref; k += nthr) sm.refind[k] = sm.pool[sm.ntr[k]];
    const int nud0 = block_compact(nhi, [&](int cidx) { return y[cidx] < 0; }, sm.ntr, sm.misc);
    for (int k = tid; k < nud0; k += nthr) sm.udets0[k] = sm.hi[sm.ntr[k]];
    const int nut = block_compact(npool, [&](int i) { return x[i] < 0 && sm.pstate[i] == ST_TRACKED; }, sm.ut, sm.misc);
    const int nmatch0 = npool - block_compact(npool, [&](int i) { return x[i] < 0; }, sm.ntr, sm.misc);
    for (int k = tid; k < npool; k += nthr) {
        const int xx = x[k];
        sm.ntr[k] = xx >= 0 ? sm.hi[xx] : -1;
        sm.used[k] = sm.pstate[k] == ST_TRACKED ? 0 : 1;
    }
    __syncthreads();
    cb_apply<T>(c, sm.pool, npool, dets, sm.ntr, sm.used);
    B2T_PHASE(6);

    // ---- stage 2: still-unmatched Tracked rows, motion_state2 x every stage-1 leftover's level-2 buffer, threshold 0.5 (:278-298)
    for (int k = tid; k < nut; k += nthr) sm.nlo[k] = sm.pool[sm.ut[k]];
    __syncthreads();
    cb_fill_ms<T>(v, CB_MS2, sm.nlo, nut, sm.rowbox);
    for (int k = tid; k < nud0; k += nthr)
        for (int q = 0; q < 4; ++q) sm.colbox[4 * k + q] = (T)buf2[4 * sm.udets0[k] + q];
    __syncthreads();
    associate<T>(c, nut, nud0, (T)p.t2, err, nullptr);
    // step 4 (:324-331): u_tracks1 become Lost with time_since_update = frame - end_frame, or Removed past max_time_lost
    const int nl = block_compact(nut, [&](int i) { return x[i] < 0; }, sm.ntr, sm.misc);
    for (int k = tid; k < nl; k += nthr) {
        const int s = sm.nlo[sm.ntr[k]];
        const int tsu = f - v.frame_id[s];
        if (tsu > p.max_time_lost) { v.state[s] = ST_REMOVED; if (v.removed_at[s] == 0) v.removed_at[s] = f; }
        else { v.state[s] = ST_LOST; v.mean[(size_t)s * 8 + CB_TSU] = (T)tsu; }
    }
    __syncthreads();
    const int nlostnow = block_compact(nl, [&](int k) { return v.state[sm.nlo[sm.ntr[k]]] == ST_LOST; }, sm.ut, sm.misc);
    for (int k = tid; k < nlostnow; k += nthr) sm.lost_now[k] = sm.nlo[sm.ntr[sm.ut[k]]];
    __syncthreads();
    // stage-2 leftovers, in column order (u_dets1)
    const int nud1 = block_compact(nud0, [&](int cidx) { return y[cidx] < 0; }, sm.ut, sm.misc);
    for (int k = tid; k < nud1; k += nthr) sm.births[k] = sm.udets0[sm.ut[k]];
    for (int k = tid; k < nut; k += nthr) { const int xx = x[k]; sm.ntr[k] = xx >= 0 ? sm.udets0[xx] : -1; sm.used[k] = 0; }
    __syncthreads();
    cb_apply<T>(c, sm.nlo, nut, dets, sm.ntr, sm.used);
    for (int k = tid; k < nud1; k += nthr) sm.udets0[k] = sm.births[k];
    __syncthreads();

    B2T_PHASE(7);
    // ---- stage 3': unconfirmed motion_state1 x the stage-2 leftovers' level-1 buffers, threshold 0.7 (:300-314)
    cb_fill_ms<T>(v, CB_MS1, sm.unconf, nunc, sm.rowbox);
    for (int k = tid; k < nud1; k += nthr)
        for (int q = 0; q < 4; ++q) sm.colbox[4 * k + q] = (T)buf1[4 * sm.udets0[k] + q];
    __syncthreads();
    associate<T>(c, nunc, nud1, (T)p.t3, err, nullptr);
    for (int k = tid; k < nunc; k += nthr)
        if (x[k] < 0) { const int s = sm.unconf[k]; v.state[s] = ST_REMOVED; if (v.removed_at[s] == 0) v.removed_at[s] = f; }
    int nbirth = block_compact(nud1, [&](int k) { return y[k] < 0 && dets[6 * sm.udets0[k] + 4] > p.new_thresh; }, sm.ntr, sm.misc);
    for (int k = tid; k < nbirth; k += nthr) sm.births[k] = sm.udets0[sm.ntr[k]];      // det indices
    __syncthreads();
    for (int k = tid; k < nunc; k += nthr) { const int xx = x[k]; sm.ntr[k] = xx < 0 ? -1 : sm.udets0[xx]; sm.used[k] = 0; }
    __syncthreads();
    cb_apply<T>(c, sm.unconf, nunc, dets, sm.ntr, sm.used);

    B2T_PHASE(8);
    // ---- births (C_BIoUSTrack.__init__ + activate, :18-46, :76-87)
    const int nfree = v.ctrl[CTRL_NFREE];
    if (nbirth > nfree) { if (tid == 0) *err |= ERR_SLOTS; nbirth = nfree; }
    const int id0 = v.ctrl[CTRL_NEXT_ID];
    for (int k = tid; k < nbirth; k += nthr) {
        const int d = sm.births[k];
        const int s = v.freelist[k];
        const float* dd = dets + 6 * d;
        T* rm = v.mean + (size_t)s * 8;
        T* rc = v.cov + (size_t)s * 64;
        float t[4], b[4];
        cb_det_tlwh(dd, t);
        cb_store4(rc + CB_HIST, t);
        cb_level1(t, b); cb_store4(rc + CB_MS1, b);
        cb_level2(t, b); cb_store4(rc + CB_MS2, b);
        rm[CB_LEN] = (T)1; rm[CB_TSU] = (T)0;
        v.tid[s] = id0 + 1 + k;
        v.state[s] = ST_TRACKED;
        v.activated[s] = (f == 1) ? 1 : 0;
        v.tracklet_len[s] = 0;
        v.start_frame[s] = f; v.frame_id[s] = f;
        v.flags[s] = 0;
        v.removed_at[s] = 0;
        v.cls[s] = dd[5]; v.score[s] = dd[4];
    }
    __syncthreads();
    for (int k = tid; k < nbirth; k += nthr) sm.births[k] = v.freelist[k];               // now slots
    if (tid == 0) v.ctrl[CTRL_NEXT_ID] = id0 + nbirth;
    __syncthreads();

    B2T_PHASE(9);
    // lost tracks are never pruned (step 4 only visits tracks that were Tracked at frame start): no P8 here
    auto last_box = [&](int s, bool tlbr, T* box) {
        const T* h = v.cov + (size_t)s * 64 + CB_HIST + 4 * ((int)v.mean[(size_t)s * 8 + CB_LEN] - 1);
        if (tlbr) cb_tlbr<T>(h, box);
        else for (int q = 0; q < 4; ++q) box[q] = h[q];
    };
    const FrameLists fl = finish_lists<T>(c, last_box, n_tracked0, n_lost0, nbirth, nref, nlostnow, out, out_rows, err, stat, tprev);
    if (tid == 0) {
        v.ctrl[CTRL_NTRACKED] = fl.nt; v.ctrl[CTRL_NLOST] = fl.nl; v.ctrl[CTRL_NFREE] = fl.nfree; v.ctrl[CTRL_ERR] = *err;
        stat[STAT_NOUT] = fl.nout; stat[STAT_NEXT_ID] = v.ctrl[CTRL_NEXT_ID]; stat[STAT_NTRACKED] = fl.nt; stat[STAT_NLOST] = fl.nl;
        stat[STAT_ERR] = *err; stat[STAT_FRAME] = f; stat[STAT_NPOOL] = npool; stat[STAT_NBIRTH] = nbirth;
        stat[STAT_NHI] = nhi; stat[STAT_NLO] = 0; stat[STAT_NEDGE] = sm.misc[50]; stat[STAT_NMATCH0] = nmatch0;
    }
}

// Shared memory of the C-BIoU step: the common arena of StepSmem.  Both detection buffer levels (2 x 4 float32 per detection) fit
// in its fp64 detbox array, so C-BIoU takes exactly the bytes of the fp64 Kalman kinds and the same shared-memory edge mirror.
inline size_t cbiou_smem_bytes(int cap, int dmax, int esm) { return StepSmem<double>::bytes(cap, dmax, esm); }
inline int cbiou_fit_esm(int cap, int dmax, int ecap, size_t limit) { return StepSmem<double>::fit_esm(cap, dmax, ecap, limit); }

}  // namespace b2t
