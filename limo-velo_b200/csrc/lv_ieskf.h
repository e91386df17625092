/*
 * lv_ieskf.h — one evaluation of the iterated error-state Kalman update, host+device.
 *
 * Replaces the body of esekf::update_iterated_dyn_share_modified
 * (include/IKFoM/IKFoM_toolkit/esekfom/esekfom.hpp:1620-1823) for n = 23, measurement block 12,
 * in the only branch LIMO-Velo can define (Nm >= 23, esekfom.hpp:1720-1729).  The 23x23 algebra
 * that the reference runs on the host between two h_dyn_share calls runs here as ONE thread block
 * between two measure-kernel launches, so a whole <= (MAX_NUM_ITERS+1)-evaluation update needs no
 * host round trip.
 *
 * The code is written as "parallel phases": LV_PAR(i, n) distributes n independent items over the
 * block and ex.sync() separates phases.  With ExecSerial (one thread, no-op sync) the very same
 * code runs on the host; tests/cpu_shim uses that to unit-test it without a GPU.
 */
#ifndef LV_IESKF_H_
#define LV_IESKF_H_

#include "lv_point_math.h"

namespace lv {

#ifndef LV_TK
#define LV_TK(k)            /* same, stamped by whichever thread runs the statement */
#endif
#ifndef LV_CK
#define LV_CK(k)            /* phase clock of the tuning build (-DLV_STEP_TIMING), see lv_measure.cu */
#endif

enum { kN = 23, kAug = 46, kMaxEvals = 8 };

struct IeskfParams {
    double R;                 /* LiDAR_noise            (Localizator.cpp:132)   */
    double D;                 /* degeneracy_threshold   (Localizator.cpp:132)   */
    double limits[kN];        /* LIMITS                 (Localizator.cpp:115)   */
    int32_t max_iter;         /* MAX_NUM_ITERS          (Localizator.cpp:114)   */
    int32_t estimate_extrinsics;
};

/* mirrors lv_iter_log of the C ABI (include/limovelo_b200.h) */
struct IterLog {
    int64_t n_matches;
    int32_t converged;
    int32_t degenerate;
    double HTH[144];
    double HTh[12];
    double dx[kN];
    double x_after[kStateLen];
};

/* ieskf_prepare() -> ieskf_step(): the part of an evaluation that depends on the iterate only */
struct StepPrep {
    double P_j[kN * kN];      /* P_ after the J blocks (esekfom.hpp:1655-1697)           */
    double dx_new[kN];        /* J * (x [-] x_prop)                                      */
    double P11inv[144];       /* P_j[:12, :12]^-1                                        */
    double T[11 * 12];        /* P_j[12:, :12] P_j[:12, :12]^-1                          */
};

/* device-resident state of one update, shared by the measure and the step kernels */
struct UpdateCtrl {
    int32_t iter;             /* loop variable i of esekfom.hpp:1634, starts at -1       */
    int32_t t;                /* number of converged evaluations (esekfom.hpp:1757)      */
    int32_t done;             /* 1: update finished, later launches return immediately   */
    int32_t status;           /* lv_status                                               */
    int32_t n_evals;
    int32_t pad_[3];
    double x_prop[kStateLen];
    double P_prop[kN * kN];
    double x[kStateLen];      /* current iterate; final state when done                  */
    double P[kN * kN];        /* final covariance when done                              */
    Frame frame;              /* transforms of the current iterate for the next measure  */
    IterLog logs[kMaxEvals];
    /* last, so that the host's read-back of the results (everything before it) leaves it out */
    StepPrep prep;
};

/* shared-memory workspace of ieskf_prepare() */
struct PrepWork {
    double x[kStateLen], xp[kStateLen];
    double P[kN * kN];
    double dx[kN], dx_new[kN];
    double J[3][9];
    double M[12 * 24];        /* [P_j11 | I] -> [. | P_j11^-1]                           */
};

/* shared-memory workspace of the step */
struct IeskfWork {
    double x[kStateLen], xp[kStateLen];
    StepPrep p;               /* copy of ieskf_prepare()'s output                        */
    double M[12 * 25];        /* [R P_j11^-1 + Q | Q | HTh] -> [. | Z]                   */
    double Kx[kN * 12];
    double Kh[kN];
    double HTH[144], HTh[12];
    double dxs[kN], dnd[kN];  /* dx_ (solved), masked */
    double J[3][9];           /* J blocks: SO3@3, SO3@6 (3x3), S2@21 (2x2 in the first 4) */
    double L[kN * kN];
    double xn[kStateLen];     /* x [+] dx_ while x is still needed                        */
    Rt32 X, IL;               /* float pose and extrinsics of xn (make_frame)             */
    int64_t n_matches;
    int32_t finish;
    int32_t degen;
    int32_t eval_idx;         /* index of this evaluation's log entry                     */
    int32_t n_evals, t, iter; /* c->n_evals, c->t, c->iter at entry                       */
};

/* executors of the "parallel phases" below: ExecSerial (host, one thread) and ExecBlock (device).
 * solve_spd12(M, w): M = [A | B] (12 rows, w <= 32 columns, row-major) with A symmetric positive definite; on return
 * the columns 12..w-1 hold A^-1 B.  Gauss-Jordan elimination without pivoting: for SPD A the pivots are those of its
 * LDL^T factorisation, all positive, and the elimination does not grow the entries, so it needs no pivot search and no
 * row swap.  Called by every thread of the block. */
struct ExecSerial {
    int tid, nthreads;
    LV_HD ExecSerial() : tid(0), nthreads(1) {}
    LV_HD void sync() {}
    LV_HD bool is_task(int) const { return true; }
    /* the same operations in the same order as ExecBlock::solve_spd12, column by column */
    LV_HD void solve_spd12(double* M, int w) {
        for (int k = 0; k < 12; ++k) {
            double m[12];
            for (int i = 0; i < 12; ++i) m[i] = M[i * w + k];
            const double ipv = 1.0 / m[k];
            for (int j = 0; j < w; ++j) {
                const double ck = M[k * w + j] * ipv;
                M[k * w + j] = ck;
                for (int i = 0; i < 12; ++i)
                    if (i != k) M[i * w + j] -= m[i] * ck;
            }
        }
    }
};
#if defined(__CUDACC__)
/* One thread block runs the step.  (A single-warp variant of the whole step was measured slower, 59 us vs
 * 45 us per evaluation: 15 k dependent fp64 / shared-memory instructions issue at ~8 cycles each when one
 * warp has nothing else to switch to.  What does pay is giving each independent serial piece its own warp
 * and keeping the 12-row elimination inside one warp's registers, see solve_spd12.) */
struct ExecBlock {
    int tid, nthreads;
    __device__ __forceinline__ ExecBlock() : tid(threadIdx.x), nthreads(blockDim.x) {}
    __device__ __forceinline__ void sync() { __syncthreads(); }
    __device__ __forceinline__ bool is_task(int k) const { return tid == 32 * k; }
    /* warp 0, lane j holds column j in 12 registers; the pivot and the multipliers of step k come from lane k by shuffle.
     * The 12 steps are unrolled so that every register index is static.  Ends with a block barrier. */
    __device__ __forceinline__ void solve_spd12(double* M, int w) {
        if (tid < 32) {
            const int lane = tid;
            const unsigned full = 0xffffffffu;
            double col[12];
#pragma unroll
            for (int i = 0; i < 12; ++i) col[i] = lane < w ? M[i * w + lane] : 0.0;
            if (lane == 0) LV_TK(48);
#pragma unroll
            for (int k = 0; k < 12; ++k) {
                const double ipv = 1.0 / __shfl_sync(full, col[k], k);
                const double ck = col[k] * ipv;
                col[k] = ck;
#pragma unroll
                for (int i = 0; i < 12; ++i)
                    if (i != k) col[i] -= __shfl_sync(full, col[i], k) * ck;
            }
            if (lane == 0) LV_TK(49);
#pragma unroll
            for (int i = 0; i < 12; ++i)
                if (lane >= 12 && lane < w) M[i * w + lane] = col[i];
            if (lane == 0) LV_TK(52);
        }
        __syncthreads();
    }
};
#endif

#define LV_PAR(i, n) for (int i = ex.tid; i < (n); i += ex.nthreads)

/* The three manifold blocks of the error state: SO3 @3, SO3 @6 (3x3), S2 @21 (2x2 in J[2][0:4]) */
LV_HD int jblock_idx(int b) { return b < 2 ? 3 + 3 * b : 21; }
LV_HD int jblock_dim(int b) { return b < 2 ? 3 : 2; }

/* for each block b: rows idx_b.. of dst (all `cols` columns) = J_b * the same rows of src.  The three row
 * sets are disjoint, so one phase serves all blocks (esekfom.hpp:1655-1697 walks them one after another). */
template <class Ex>
LV_HD void apply_rows3(Ex& ex, double* dst, const double* src, const double (*J)[9], int cols, int stride) {
    LV_PAR(it, 3 * cols) {
        const int b = it / cols, i = it - b * cols;
        const int idx = jblock_idx(b), d = jblock_dim(b);
        double v[3], r[3];
        for (int c = 0; c < d; ++c) v[c] = src[(idx + c) * stride + i];
        for (int a = 0; a < d; ++a) {
            double s = 0;
            for (int c = 0; c < d; ++c) s += J[b][a * d + c] * v[c];
            r[a] = s;
        }
        for (int a = 0; a < d; ++a) dst[(idx + a) * stride + i] = r[a];
    }
}
/* for each block b: columns idx_b.. of M (all `rows` rows) = the same columns * J_b^T */
template <class Ex>
LV_HD void apply_cols3(Ex& ex, double* M, const double (*J)[9], int rows, int stride) {
    LV_PAR(it, 3 * rows) {
        const int b = it / rows, i = it - b * rows;
        const int idx = jblock_idx(b), d = jblock_dim(b);
        double v[3], r[3];
        for (int c = 0; c < d; ++c) v[c] = M[i * stride + idx + c];
        for (int a = 0; a < d; ++a) {
            double s = 0;
            for (int c = 0; c < d; ++c) s += v[c] * J[b][a * d + c];
            r[a] = s;
        }
        for (int a = 0; a < d; ++a) M[i * stride + idx + a] = r[a];
    }
}

/* ---- serial helpers for the (rare) degenerate branch, esekfom.hpp:1736-1744 ---------------- */
/* cyclic Jacobi, eigenvalues ascending, vectors = columns of V, largest component positive.
 * The reference uses Eigen::EigenSolver whose pair order is unspecified: the degenerate branch
 * is "parity unpinned" (DESIGN.md).                                                           */
LV_HD_COLD void sym_eig6(const double* Ain, double* ev, double* V) {
    const int n = 6;
    double A[36];
    for (int i = 0; i < 36; ++i) { A[i] = Ain[i]; V[i] = (i % 7 == 0) ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0, diag = 0;
        for (int i = 0; i < n; ++i) {
            diag += A[i * n + i] * A[i * n + i];
            for (int j = i + 1; j < n; ++j) off += A[i * n + j] * A[i * n + j];
        }
        if (off <= 1e-30 * diag || off == 0.0) break;
        for (int p = 0; p < n; ++p)
            for (int q = p + 1; q < n; ++q) {
                const double apq = A[p * n + q];
                if (apq == 0.0) continue;
                const double theta = (A[q * n + q] - A[p * n + p]) / (2 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1));
                const double c = 1 / sqrt(t * t + 1), s = t * c;
                for (int k = 0; k < n; ++k) {
                    const double akp = A[k * n + p], akq = A[k * n + q];
                    A[k * n + p] = c * akp - s * akq;
                    A[k * n + q] = s * akp + c * akq;
                }
                for (int k = 0; k < n; ++k) {
                    const double apk = A[p * n + k], aqk = A[q * n + k];
                    A[p * n + k] = c * apk - s * aqk;
                    A[q * n + k] = s * apk + c * aqk;
                }
                for (int k = 0; k < n; ++k) {
                    const double vkp = V[k * n + p], vkq = V[k * n + q];
                    V[k * n + p] = c * vkp - s * vkq;
                    V[k * n + q] = s * vkp + c * vkq;
                }
            }
    }
    /* selection sort of the eigenpairs (ascending) + sign normalisation */
    double Vs[36];
    bool used[6] = {false, false, false, false, false, false};
    for (int j = 0; j < n; ++j) {
        int src = -1;
        for (int c = 0; c < n; ++c)
            if (!used[c] && (src < 0 || A[c * n + c] < A[src * n + src])) src = c;
        used[src] = true;
        ev[j] = A[src * n + src];
        int imax = 0;
        for (int k = 1; k < n; ++k)
            if (fabs(V[k * n + src]) > fabs(V[imax * n + src])) imax = k;
        const double sg = V[imax * n + src] < 0 ? -1.0 : 1.0;
        for (int k = 0; k < n; ++k) Vs[k * n + j] = sg * V[k * n + src];
    }
    for (int i = 0; i < 36; ++i) V[i] = Vs[i];
}

/* dnd[0:6] = V^-1 * sel * dx_[0:6]  (esekfom.hpp:1736-1744), executed by one thread */
LV_HD_COLD void degenerate_mask(const double* HTH, double D, const double* dxs, double* dnd) {
    double A6[36], ev[6], V[36], sel[36];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j < 6; ++j) A6[i * 6 + j] = HTH[i * 12 + j];
    sym_eig6(A6, ev, V);
    double prod = 1;
    for (int i = 0; i < 6; ++i) prod *= ev[i];
    if (prod < 1e-20)
        for (int i = 0; i < 36; ++i) V[i] = (i % 7 == 0) ? 1.0 : 0.0;
    for (int i = 0; i < 36; ++i) sel[i] = V[i];
    for (int j = 0; j < 6; ++j)
        if (ev[j] < D)
            for (int c = 0; c < 6; ++c) sel[j * 6 + c] = 0;
    double t[6];
    for (int i = 0; i < 6; ++i) {
        double s = 0;
        for (int j = 0; j < 6; ++j) s += sel[i * 6 + j] * dxs[j];
        t[i] = s;
    }
    /* solve V y = t by Gauss-Jordan with partial pivoting (== V^-1 t) */
    double M[6 * 7];
    for (int i = 0; i < 6; ++i) {
        for (int j = 0; j < 6; ++j) M[i * 7 + j] = V[i * 6 + j];
        M[i * 7 + 6] = t[i];
    }
    for (int k = 0; k < 6; ++k) {
        int p = k;
        for (int i = k + 1; i < 6; ++i)
            if (fabs(M[i * 7 + k]) > fabs(M[p * 7 + k])) p = i;
        if (p != k)
            for (int j = 0; j < 7; ++j) { const double tmp = M[k * 7 + j]; M[k * 7 + j] = M[p * 7 + j]; M[p * 7 + j] = tmp; }
        const double pv = M[k * 7 + k];
        for (int j = k; j < 7; ++j) M[k * 7 + j] /= pv;
        for (int i = 0; i < 6; ++i) {
            if (i == k) continue;
            const double f = M[i * 7 + k];
            for (int j = k; j < 7; ++j) M[i * 7 + j] -= f * M[k * 7 + j];
        }
    }
    for (int i = 0; i < 6; ++i) dnd[i] = M[i * 7 + 6];
}

/* true iff every eigenvalue of HTH[0:6,0:6] exceeds D: Cholesky of (A - D I) succeeds */
LV_HD bool all_eigs_above(const double* HTH, double D) {
    double Lc[36];
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) {
            double s = HTH[i * 12 + j] - (i == j ? D : 0.0);
            for (int k = 0; k < j; ++k) s -= Lc[i * 6 + k] * Lc[j * 6 + k];
            if (i == j) {
                if (!(s > 0.0)) return false;
                Lc[i * 6 + i] = sqrt(s);
            } else {
                Lc[i * 6 + j] = s / Lc[j * 6 + j];
            }
        }
    return true;
}

/* J block of manifold block b for the error-state vector d (esekfom.hpp:1655-1697, 1770-1812):
 * SO3: A(d_b)^T ; S2: Nx(grav_now) * Mx(grav_prop, d_b).  LV_HD_COLD: one copy of the trig code. */
LV_HD_COLD void jblock(int b, const double* d, const double* x_now, const double* x_prop, double* J) {
    if (b < 2) {
        const Mat3d Jt = mat3_transpose(A_matrix(load_vec3(d + 3 + 3 * b)));
        for (int i = 0; i < 9; ++i) J[i] = Jt.m[i];
    } else {
        s2_J(load_vec3(x_now + kGrav), load_vec3(x_prop + kGrav), d[21], d[22], J);
    }
}

/* the degenerate case of one evaluation, one thread: w->dnd = the masked dx_, w->xn = x [+] dnd, the frame of xn */
LV_HD_COLD void degenerate_redo(double D, IeskfWork* w, Frame* frame) {
    degenerate_mask(w->HTH, D, w->dxs, w->dnd);
    for (int i = 0; i < kStateLen; ++i) w->xn[i] = w->x[i];
    state_boxplus(w->xn, w->dnd);
    make_frame(w->xn, frame);
}

/*
 * The iterate-only part of an evaluation (esekfom.hpp:1651-1697): dx = x [-] x_prop, the J blocks,
 * dx_new = J dx and P_ = J P_prop J^T, and what the gain of ieskf_step() needs of P_: P_11^-1 and T = P_21 P_11^-1.
 * Nothing here depends on the measurement, so on the device it runs in a spare block of the fit kernel, beside the
 * measurement of the same iterate, and hands its results to the step through c->prep.  Independent serial pieces
 * are "tasks": on the device each runs in its own warp (ex.is_task, tasks 0..3 need >= 128 threads), on the host
 * one after another.
 */
template <class Ex>
LV_HD_NOINLINE void ieskf_prepare(Ex& ex, UpdateCtrl* c, PrepWork* w) {
    const int n = kN;
    StepPrep* out = &c->prep;
    LV_PAR(i, n * n) w->P[i] = c->P_prop[i];
    LV_PAR(i, kStateLen) { w->x[i] = c->x[i]; w->xp[i] = c->x_prop[i]; }
    ex.sync();
    for (int b = 0; b < 3; ++b)
        if (ex.is_task(b)) {
            const int idx = jblock_idx(b), d = jblock_dim(b);
            if (b < 2) {
                const int q = b == 0 ? kRot : kOffR;
                store_vec3(w->dx + idx, so3_log(quat_mul(quat_conj(load_quat(w->xp + q)), load_quat(w->x + q))));
            } else {
                s2_boxminus(load_vec3(w->x + kGrav), load_vec3(w->xp + kGrav), w->dx + 21);
            }
            jblock(b, w->dx, w->x, w->xp, w->J[b]);
            for (int a = 0; a < d; ++a) {
                double s = 0;
                for (int k = 0; k < d; ++k) s += w->J[b][a * d + k] * w->dx[idx + k];
                w->dx_new[idx + a] = s;
            }
        }
    if (ex.is_task(3)) {
        const int lin[5][2] = {{0, kPos}, {9, kOffT}, {12, kVel}, {15, kBg}, {18, kBa}};
        for (int g = 0; g < 5; ++g)
            for (int i = 0; i < 3; ++i) {
                const double v = w->x[lin[g][1] + i] - w->xp[lin[g][1] + i];
                w->dx[lin[g][0] + i] = v;
                w->dx_new[lin[g][0] + i] = v;
            }
    }
    ex.sync();
    apply_rows3(ex, w->P, w->P, w->J, n, n);
    ex.sync();
    apply_cols3(ex, w->P, w->J, n, n);
    ex.sync();
    LV_PAR(it, 12 * 24) {
        const int i = it / 24, j = it - i * 24;
        w->M[it] = j < 12 ? w->P[i * n + j] : (j - 12 == i ? 1.0 : 0.0);
    }
    LV_PAR(i, n * n) out->P_j[i] = w->P[i];
    LV_PAR(i, n) out->dx_new[i] = w->dx_new[i];
    ex.sync();
    ex.solve_spd12(w->M, 24);
    LV_PAR(i, 144) out->P11inv[i] = w->M[(i / 12) * 24 + 12 + i % 12];
    LV_PAR(it, 11 * 12) {
        const int i = it / 12, j = it - i * 12;
        double s = 0;
        for (int k = 0; k < 12; ++k) s += w->P[(12 + i) * n + k] * w->M[k * 24 + 12 + j];
        out->T[it] = s;
    }
}

/* global -> workspace copies of one evaluation; no barrier inside (the caller's next barrier covers them) */
template <class Ex>
LV_HD void ieskf_load(Ex& ex, const UpdateCtrl* c, IeskfWork* w) {
    LV_PAR(i, (int)(sizeof(StepPrep) / sizeof(double))) reinterpret_cast<double*>(&w->p)[i] = reinterpret_cast<const double*>(&c->prep)[i];
    LV_PAR(i, kStateLen) { w->x[i] = c->x[i]; w->xp[i] = c->x_prop[i]; }
    if (ex.tid == 0) {
        w->n_evals = c->n_evals;
        w->eval_idx = w->n_evals < kMaxEvals ? w->n_evals : kMaxEvals - 1;
        w->t = c->t;
        w->iter = c->iter;
    }
}

/*
 * One evaluation (esekfom.hpp:1699-1822) after ieskf_prepare().  Inputs: ieskf_load() done, w->HTH/HTh/n_matches
 * reduced, all visible (a barrier after both).  Outputs: c->x (new iterate), c->frame, c->logs[], and on exit
 * c->P, c->done.
 */
template <class Ex>
LV_HD_NOINLINE void ieskf_step(Ex& ex, const IeskfParams& prm, UpdateCtrl* c, IeskfWork* w) {
    const int n = kN;
    const double* dx_new = w->p.dx_new;
    IterLog* lg = &c->logs[w->eval_idx];
    /* Nm < n: the reference takes esekfom.hpp:1701-1709 and then reads an uninitialised HTH
     * (SURVEY 8c quirk 4).  Here: stop, report LV_TOO_FEW_MATCHES, keep the current iterate. */
    if (w->n_matches < n) {
        if (ex.tid == 0) {
            lg->n_matches = w->n_matches;
            c->status = 2; /* LV_TOO_FEW_MATCHES */
            c->done = 1;
        }
        return;
    }
    LV_CK(3);

    /* Gain (esekfom.hpp:1722-1729), information form.  The reference forms P_inv = ((P/R)^-1 + E^T Q E)^-1 with two
     * 23x23 inverses (Q = HTH, E = [I12 0]) and uses only P_inv[:, :12].  With S = P/R and S11 invertible the
     * matrix-inversion lemma gives, also for singular Q (estimate_extrinsics = false),
     *   P_inv[:, :12] = S[:, :12] (I12 + Q S11)^-1 = [I ; T] (S11^-1 + Q)^-1,   T = S21 S11^-1 = P21 P11^-1.
     * A = S11^-1 + Q = R P11^-1 + Q is symmetric positive definite, so one 12x12 SPD system with 13 right-hand sides
     * replaces both inverses:  Z = A^-1 [Q | HTh],  K_x[:, :12] = [Z_Q ; T Z_Q],  K_h = [Z_h ; T Z_h].  P11^-1 and T
     * depend on the iterate only and come from ieskf_prepare() (DESIGN.md, "gain formulation").                     */
    LV_PAR(it, 12 * 25) {
        const int i = it / 25, j = it - i * 25;
        double v;
        if (j < 12) v = prm.R * w->p.P11inv[i * 12 + j] + w->HTH[i * 12 + j];
        else if (j < 24) v = w->HTH[i * 12 + (j - 12)];
        else v = w->HTh[i];
        w->M[it] = v;
    }
    ex.sync();
    LV_CK(5);
    if (ex.is_task(1)) { LV_TK(50); w->degen = all_eigs_above(w->HTH, prm.D) ? 0 : 1; LV_TK(51); }   /* beside the solve (warp 1) */
    ex.solve_spd12(w->M, 25);
    LV_CK(6);
    LV_PAR(it, n * 13) {
        const int i = it / 13, j = it - i * 13;
        double s;
        if (i < 12) {
            s = w->M[i * 25 + 12 + j];
        } else {
            s = 0;
            for (int k = 0; k < 12; ++k) s += w->p.T[(i - 12) * 12 + k] * w->M[k * 25 + 12 + j];
        }
        if (j < 12) w->Kx[i * 12 + j] = s; else w->Kh[i] = s;
    }
    ex.sync();
    /* dx_ = K_h + (K_x - I) dx_new   (esekfom.hpp:1733) */
    LV_PAR(i, n) {
        double s = 0;
        for (int j = 0; j < 12; ++j) s += w->Kx[i * 12 + j] * dx_new[j];
        w->dxs[i] = w->Kh[i] + s - dx_new[i];
        w->dnd[i] = w->dxs[i];
    }
    ex.sync();
    LV_CK(7);

    /* x [+]= dx_ (esekfom.hpp:1747), assuming the non-degenerate case (the test of :1736-1744 ran beside the
     * solve); the rare degenerate case redoes the update below.  make_frame() (State.cpp:51-62) is split over
     * tasks 0 and 1 (pose, extrinsics) and composed by task 0 after the barrier. */
    LV_PAR(i, 144) lg->HTH[i] = w->HTH[i];
    LV_PAR(i, 12) lg->HTh[i] = w->HTh[i];
    LV_PAR(i, n) lg->dx[i] = w->dxs[i];
    LV_TK(24 + (ex.tid >> 5));
#pragma unroll 1
    for (int b = 0; b < 2; ++b)
        if (ex.is_task(b)) {   /* b = 0: pose (rot @3, pos @0), b = 1: extrinsics (offset_R @6, offset_T @9) */
            const int qo = b == 0 ? kRot : kOffR, to = b == 0 ? kPos : kOffT;
            for (int i = 0; i < 3; ++i) w->xn[to + i] = w->x[to + i] + w->dnd[9 * b + i];
            const Quatd q = quat_mul(load_quat(w->x + qo), so3_exp(load_vec3(w->dnd + 3 + 3 * b), 0.5));
            store_quat(w->xn + qo, q);
            const Mat3d R = quat_to_rot(q), Ri = quat_to_rot(quat_conj(q));
            Rt32& X = b == 0 ? w->X : w->IL;
            for (int i = 0; i < 9; ++i) X.R[i] = (float)R.m[i];
            for (int i = 0; i < 3; ++i) X.t[i] = (float)w->xn[to + i];
            double* dst = b == 0 ? c->frame.R_inv : c->frame.RLI_inv;
            for (int i = 0; i < 9; ++i) dst[i] = Ri.m[i];
        }
    if (ex.is_task(2)) store_vec3(w->xn + kGrav, s2_boxplus(load_vec3(w->x + kGrav), w->dnd[21], w->dnd[22]));
    if (ex.is_task(3)) {
        for (int i = 0; i < 9; ++i) w->xn[kVel + i] = w->x[kVel + i] + w->dnd[12 + i];   /* vel, bg, ba */
        int conv = 1;                                              /* :1748-1756 uses dx_ (pre-mask) */
        for (int i = 0; i < n; ++i)
            if (fabs(w->dxs[i]) > prm.limits[i]) { conv = 0; break; }
        const int t = w->t + conv;                                 /* :1757 */
        if (!t && w->iter == prm.max_iter - 2) conv = 1;           /* :1759-1762 */
        lg->n_matches = w->n_matches;
        lg->converged = conv;
        c->t = t;
        c->n_evals = w->n_evals + 1;
        w->finish = (t > 1 || w->iter == prm.max_iter - 1) ? 1 : 0;   /* :1764 */
        c->iter = w->iter + 1;
    }
    if ((ex.tid & 31) == 0 && ex.tid < 160) LV_TK(32 + (ex.tid >> 5));
    ex.sync();
    if (ex.is_task(0)) {
        c->frame.lidar_to_world = rt_mul(w->X, w->IL);
        c->frame.world_to_lidar = rt_mul(rt_inv(w->IL), rt_inv(w->X));
        c->frame.lidar_to_imu = w->IL;
    }
    if (w->degen) {        /* esekfom.hpp:1736-1744: mask dx_[0:6] and redo the boxplus serially */
        if (ex.tid == 0) degenerate_redo(prm.D, w, &c->frame);
        ex.sync();
    }
    if (ex.is_task(1)) lg->degenerate = w->degen;
    LV_PAR(i, kStateLen) {
        const double v = w->xn[i];
        w->x[i] = v;
        c->x[i] = v;
        lg->x_after[i] = v;
    }
    ex.sync();
    LV_CK(8);
    if (!w->finish) return;

    /* exit block, esekfom.hpp:1766-1817 */
    double* Pj = w->p.P_j;
    LV_PAR(i, n * n) w->L[i] = Pj[i];
    for (int b = 0; b < 3; ++b)
        if (ex.is_task(b)) jblock(b, w->dxs, w->x, w->xp, w->J[b]);
    ex.sync();
    apply_rows3(ex, w->L, Pj, w->J, n, n);
    apply_rows3(ex, w->Kx, w->Kx, w->J, 12, 12);
    ex.sync();
    apply_cols3(ex, w->L, w->J, n, n);
    apply_cols3(ex, Pj, w->J, n, n);
    ex.sync();
    LV_PAR(it, n * n) {                                            /* :1817 */
        const int i = it / n, j = it - i * n;
        double s = 0;
        for (int k = 0; k < 12; ++k) s += w->Kx[i * 12 + k] * Pj[k * n + j];
        c->P[it] = w->L[it] - s;
    }
    if (ex.tid == 0) c->done = 1;
    ex.sync();
    LV_CK(9);
}

/* start of an update: x_prop = x, P_prop = P, loop counters (esekfom.hpp:1622-1634) */
template <class Ex>
LV_HD void ieskf_begin(Ex& ex, UpdateCtrl* c) {
    LV_PAR(i, kStateLen) c->x_prop[i] = c->x[i];
    LV_PAR(i, kN * kN) c->P_prop[i] = c->P[i];
    if (ex.tid == 0) {
        c->iter = -1;
        c->t = 0;
        c->done = 0;
        c->status = 0;
        c->n_evals = 0;
        make_frame(c->x, &c->frame);
    }
    ex.sync();
}

}  // namespace lv
#endif
