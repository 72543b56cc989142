// b2k_fkj.cuh -- forward kinematics + geometric Jacobian kernels for sm_100a.
//
// Mapping (DESIGN.md "Kernel K12"): a warp owns a TILE of 32 joint configurations.  Lane l
// walks the serial chain of row (tile*32 + l) entirely in registers -- pose as four 3-vectors
// (bottom row 0 0 0 1 implied), chain constants and sincos coefficients read straight from the
// constant bank (the chain is a __grid_constant__ kernel parameter, so every folded constant is
// an immediate c[0x0][..] operand of the FMA).  The warp as a whole moves the tile's q block and
// its T / J blocks between HBM and registers through a per-warp shared-memory stage so that
// every global access is a fully coalesced warp transaction:
//     q tile  (32 x ldq)  : 16-byte cp.async (LDGSTS) straight into smem; one row per lane read back
//     T tile  (32 x 16)   : one pose row per lane, 256-bit stores straight from registers
//                           (a row is 128 B / 64 B contiguous: full sectors without staging)
//     J tile  (32 x 6n)   : registers -> 16-byte vector STS into a stage that is the exact image of
//                           the output block -> ONE TMA bulk copy (cp.async.bulk, SASS UBLKCP)
// Two forms of every walk: the general kernels (k_fkj_forward / k_fkj_backward: any row stride, jindex
// permutation, alignment, chain shape, ragged tiles) and the lean kernels (k_fkj_fast / k_fkj_back_fast)
// the launcher picks for the common call, with all of that fixed at compile time.
// No tensor cores: the products are 3x3 / 6xn (far below an MMA tile) -- this is HBM-bound
// streaming work (SURVEY.md section 8d: 520 B per evaluation for Panda fp64).
//
// Arithmetic follows reference methods.cpp:318-352 (pose) and the column rules of
// methods.cpp:137-196 (Jacobian), re-associated: constants folded per joint, pose walked
// left-to-right once, base-frame Jacobian columns formed as z_j x (p_e - p_j) instead of the
// reference's end-effector-frame walk + blkdiag(R,R) rotation.  Same values to rounding.
#pragma once

#include <type_traits>

#include "b2k_common.cuh"
#include "b2k_trig.cuh"

// pose T = [c0 c1 c2 p] (columns), all in registers
template <typename real>
struct Pose {
    real c0[3], c1[3], c2[3], p[3];
};

template <typename real>
__device__ __forceinline__ void pose_from_const(Pose<real> &T, const real *A)
{
#pragma unroll
    for (int i = 0; i < 3; i++) {
        T.c0[i] = A[i * 4 + 0];
        T.c1[i] = A[i * 4 + 1];
        T.c2[i] = A[i * 4 + 2];
        T.p[i] = A[i * 4 + 3];
    }
}

// T <- T * A for a folded constant A of structure class `kind` (uniform across the grid)
template <typename real>
__device__ __forceinline__ void pose_mul_const_right(Pose<real> &T, const real *A, int kind)
{
    if (kind & AK_TX) {
#pragma unroll
        for (int i = 0; i < 3; i++) T.p[i] = fma(T.c0[i], A[3], T.p[i]);
    }
    if (kind & AK_TY) {
#pragma unroll
        for (int i = 0; i < 3; i++) T.p[i] = fma(T.c1[i], A[7], T.p[i]);
    }
    if (kind & AK_TZ) {
#pragma unroll
        for (int i = 0; i < 3; i++) T.p[i] = fma(T.c2[i], A[11], T.p[i]);
    }
    switch (kind & AK_ROTMASK) {
    case AK_IDENT: break;
    case AK_RX:
#pragma unroll
        for (int i = 0; i < 3; i++) {
            real a = T.c1[i], b = T.c2[i];
            T.c1[i] = fma(a, A[5], b * A[9]);
            T.c2[i] = fma(a, A[6], b * A[10]);
        }
        break;
    case AK_RY:
#pragma unroll
        for (int i = 0; i < 3; i++) {
            real a = T.c0[i], b = T.c2[i];
            T.c0[i] = fma(a, A[0], b * A[8]);
            T.c2[i] = fma(a, A[2], b * A[10]);
        }
        break;
    case AK_RZ:
#pragma unroll
        for (int i = 0; i < 3; i++) {
            real a = T.c0[i], b = T.c1[i];
            T.c0[i] = fma(a, A[0], b * A[4]);
            T.c1[i] = fma(a, A[1], b * A[5]);
        }
        break;
    default:
#pragma unroll
        for (int i = 0; i < 3; i++) {
            real a = T.c0[i], b = T.c1[i], c = T.c2[i];
            T.c0[i] = fma(a, A[0], fma(b, A[4], c * A[8]));
            T.c1[i] = fma(a, A[1], fma(b, A[5], c * A[9]));
            T.c2[i] = fma(a, A[2], fma(b, A[6], c * A[10]));
        }
        break;
    }
}

// T <- A * T (used by the backward / end-effector-frame walk and for the base)
template <typename real>
__device__ __forceinline__ void pose_mul_const_left(Pose<real> &T, const real *A, int kind)
{
    const int rk = kind & AK_ROTMASK;
    real *cols[4] = {T.c0, T.c1, T.c2, T.p};
    if (rk == AK_IDENT) {
    } else if (rk == AK_RX) { // rows 1,2 mix
#pragma unroll
        for (int j = 0; j < 4; j++) {
            real a = cols[j][1], b = cols[j][2];
            cols[j][1] = fma(A[5], a, A[6] * b);
            cols[j][2] = fma(A[9], a, A[10] * b);
        }
    } else if (rk == AK_RY) { // rows 0,2 mix
#pragma unroll
        for (int j = 0; j < 4; j++) {
            real a = cols[j][0], b = cols[j][2];
            cols[j][0] = fma(A[0], a, A[2] * b);
            cols[j][2] = fma(A[8], a, A[10] * b);
        }
    } else if (rk == AK_RZ) { // rows 0,1 mix
#pragma unroll
        for (int j = 0; j < 4; j++) {
            real a = cols[j][0], b = cols[j][1];
            cols[j][0] = fma(A[0], a, A[1] * b);
            cols[j][1] = fma(A[4], a, A[5] * b);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            real a = cols[j][0], b = cols[j][1], c = cols[j][2];
            cols[j][0] = fma(A[0], a, fma(A[1], b, A[2] * c));
            cols[j][1] = fma(A[4], a, fma(A[5], b, A[6] * c));
            cols[j][2] = fma(A[8], a, fma(A[9], b, A[10] * c));
        }
    }
    if (kind & AK_TX) T.p[0] += A[3];
    if (kind & AK_TY) T.p[1] += A[7];
    if (kind & AK_TZ) T.p[2] += A[11];
}

// rotate the column pair (a, b) <- (c a + s b, c b - s a): the right-multiplication by an
// elementary rotation about the third axis (reference rx/ry/rz, fknm.cpp:1320-1440)
template <typename real>
__device__ __forceinline__ void rot_cols(real *a, real *b, real s, real c)
{
#pragma unroll
    for (int i = 0; i < 3; i++) {
        real x = a[i], y = b[i];
        a[i] = fma(c, x, s * y);
        b[i] = fma(c, y, -(s * x));
    }
}

// T <- T * ET(eta) for a joint of the given axis (eta already sign-flipped)
template <typename real>
__device__ __forceinline__ void pose_joint_right(Pose<real> &T, int axis, real eta, const TrigC<real> &tc)
{
    if (axis < 3) {
        real s, c;
        b2k_sincos(eta, tc, &s, &c);
        if (axis == B2K_RZ) rot_cols(T.c0, T.c1, s, c);
        else if (axis == B2K_RX) rot_cols(T.c1, T.c2, s, c);
        else rot_cols(T.c2, T.c0, s, c);
    } else {
        if (axis == B2K_TX) {
#pragma unroll
            for (int i = 0; i < 3; i++) T.p[i] = fma(T.c0[i], eta, T.p[i]);
        } else if (axis == B2K_TY) {
#pragma unroll
            for (int i = 0; i < 3; i++) T.p[i] = fma(T.c1[i], eta, T.p[i]);
        } else {
#pragma unroll
            for (int i = 0; i < 3; i++) T.p[i] = fma(T.c2[i], eta, T.p[i]);
        }
    }
}

// rows (IA, IB) of all four columns: a' = c a - s b ; b' = s a + c b  (left-multiplication by
// an elementary rotation about the remaining axis)
template <typename real, int IA, int IB>
__device__ __forceinline__ void rot_rows(Pose<real> &T, real s, real c)
{
    real *cols[4] = {T.c0, T.c1, T.c2, T.p};
#pragma unroll
    for (int j = 0; j < 4; j++) {
        real x = cols[j][IA], y = cols[j][IB];
        cols[j][IA] = fma(c, x, -(s * y));
        cols[j][IB] = fma(s, x, c * y);
    }
}

// T <- ET(eta) * T
template <typename real>
__device__ __forceinline__ void pose_joint_left(Pose<real> &T, int axis, real eta, const TrigC<real> &tc)
{
    if (axis < 3) {
        real s, c;
        b2k_sincos(eta, tc, &s, &c);
        if (axis == B2K_RZ) rot_rows<real, 0, 1>(T, s, c);
        else if (axis == B2K_RX) rot_rows<real, 1, 2>(T, s, c);
        else rot_rows<real, 2, 0>(T, s, c);
    } else {
        if (axis == B2K_TX) T.p[0] += eta;
        else if (axis == B2K_TY) T.p[1] += eta;
        else T.p[2] += eta;
    }
}

// end-effector-frame Jacobian column read off U (reference methods.cpp:243-302):
// revolute about axis AX: lin = r_K1 * p_A - r_K2 * p_B, ang = r_AX, where r_k is row k of U's rotation
template <typename real, int AX>
__device__ __forceinline__ void je_col_rev(const Pose<real> &U, real sg, real *col)
{
    constexpr int K1 = (AX == 0) ? 2 : (AX == 1) ? 0 : 1;
    constexpr int K2 = (AX == 0) ? 1 : (AX == 1) ? 2 : 0;
    constexpr int PA = (AX == 0) ? 1 : (AX == 1) ? 2 : 0;
    constexpr int PB = (AX == 0) ? 2 : (AX == 1) ? 0 : 1;
    const real *cols[3] = {U.c0, U.c1, U.c2};
#pragma unroll
    for (int i = 0; i < 3; i++) {
        col[i] = sg * fma(cols[i][K1], U.p[PA], -(cols[i][K2] * U.p[PB]));
        col[3 + i] = sg * cols[i][AX];
    }
}
template <typename real, int K>
__device__ __forceinline__ void je_col_pri(const Pose<real> &U, real sg, real *col)
{
    const real *cols[3] = {U.c0, U.c1, U.c2};
#pragma unroll
    for (int i = 0; i < 3; i++) {
        col[i] = sg * cols[i][K];
        col[3 + i] = (real)0;
    }
}

// ------------------------------------------------------------------ the forward chain walk (one row, registers only)
// T = A_0 J_0(q) A_1 J_1(q) ... A_{n-1} J_{n-1}(q) A_n.  When WJ, also records for every joint the
// (signed) joint axis z_j and the joint origin p_j in the start frame, from which the base-frame
// Jacobian column is z_j x (p_e - p_j) | z_j (revolute) or z_j | 0 (prismatic).
// getq(j, col) returns this row's coordinate of joint j, stored in column col of q (shared
// memory in the FK kernels; registers, indexed by the compile-time j, in the IK kernel).
// PROF selects the code shape (uniform for the whole grid, decided on the host):
//   1 "DH-like": every joint is an unflipped Rz and every inter-joint constant has the Rx form
//     [[1,0,0],[0,a,b],[0,c,d]] (+ translation) -- standard / modified DH robots and the Panda ETS.
//     Straight-line code: no switches (the compiler if-converts small uniform switches into
//     select chains, ncu profiles/r01_fkj_v2.md), all n sincos evaluated as one interleaved batch.
//   0 generic: any axis / flip / constant, runtime (uniform) switches.
//   TRIG = 1 (the IK loop, whose iterates leave [-pi, pi] in some lanes of most warps): fp32 angles are reduced once
//   and go to the special-function unit whatever their size, so a warp never runs two sincos paths back to back.
// zj / pj are indexed zj[j][i]: register arrays real[N][3], or JRowCols views of a Jacobian row in shared memory.
template <typename real, int N, bool WJ, int PROF, int TRIG = 0, typename GetQ, typename ZJ, typename PJ>
__device__ __forceinline__ void chain_forward(const ChainP<real, N> &P, GetQ getq, Pose<real> &T, ZJ zj, PJ pj)
{
    if constexpr (PROF == 1) {
        real eta[N], sn[N], cs[N];
#pragma unroll
        for (int j = 0; j < N; j++) eta[j] = getq(j, P.jidx[j]);
        if constexpr (TRIG == 1 && sizeof(real) == 4) b2k_sincos_batch_reduced<N>(eta, sn, cs);
        else b2k_sincos_batch<real, N>(eta, P.trig, sn, cs);
        pose_from_const(T, P.A[0]);
#pragma unroll
        for (int j = 0; j < N; j++) {
            if (j > 0) {
                const real *A = P.A[j];
#pragma unroll
                for (int i = 0; i < 3; i++) {
                    T.p[i] = fma(T.c0[i], A[3], fma(T.c1[i], A[7], fma(T.c2[i], A[11], T.p[i])));
                    real a = T.c1[i], b = T.c2[i];
                    T.c1[i] = fma(a, A[5], b * A[9]);
                    T.c2[i] = fma(a, A[6], b * A[10]);
                }
            }
            if (WJ) {
#pragma unroll
                for (int i = 0; i < 3; i++) { zj[j][i] = T.c2[i]; pj[j][i] = T.p[i]; }
            }
            rot_cols(T.c0, T.c1, sn[j], cs[j]);
        }
        if (P.akind[N] != AK_IDENT) { // tail constant (tool folded in): any SE(3)
            const real *A = P.A[N];
#pragma unroll
            for (int i = 0; i < 3; i++) {
                real a = T.c0[i], b = T.c1[i], c = T.c2[i];
                T.p[i] = fma(a, A[3], fma(b, A[7], fma(c, A[11], T.p[i])));
                T.c0[i] = fma(a, A[0], fma(b, A[4], c * A[8]));
                T.c1[i] = fma(a, A[1], fma(b, A[5], c * A[9]));
                T.c2[i] = fma(a, A[2], fma(b, A[6], c * A[10]));
            }
        }
    } else {
        pose_from_const(T, P.A[0]);
#pragma unroll
        for (int j = 0; j < N; j++) {
            if (j > 0) pose_mul_const_right(T, P.A[j], P.akind[j]);
            const int ax = P.axis[j];
            real eta = getq(j, P.jidx[j]);
            const real sg = P.flip[j] ? (real)-1 : (real)1;
            eta *= sg;
            if (WJ) {
                const int k = ax < 3 ? ax : ax - 3;
#pragma unroll
                for (int i = 0; i < 3; i++) {
                    real col = (k == 0) ? T.c0[i] : (k == 1) ? T.c1[i] : T.c2[i];
                    zj[j][i] = sg * col;
                    pj[j][i] = T.p[i];
                }
            }
            pose_joint_right(T, ax, eta, P.trig);
        }
        pose_mul_const_right(T, P.A[N], P.akind[N]);
    }
}

// base-frame Jacobian row (6 x N, row-major) of one configuration from the walk's stash
template <typename real, int N, int PROF>
__device__ __forceinline__ void jacob0_row(const ChainP<real, N> &P, const Pose<real> &T, real (*zj)[3],
                                           real (*pj)[3], real *row)
{
#pragma unroll
    for (int j = 0; j < N; j++) {
        const bool rev = PROF == 1 ? true : (P.axis[j] < 3);
        if (rev) {
            real dx = T.p[0] - pj[j][0], dy = T.p[1] - pj[j][1], dz = T.p[2] - pj[j][2];
            row[0 * N + j] = fma(zj[j][1], dz, -(zj[j][2] * dy));
            row[1 * N + j] = fma(zj[j][2], dx, -(zj[j][0] * dz));
            row[2 * N + j] = fma(zj[j][0], dy, -(zj[j][1] * dx));
            row[3 * N + j] = zj[j][0];
            row[4 * N + j] = zj[j][1];
            row[5 * N + j] = zj[j][2];
        } else {
            row[0 * N + j] = zj[j][0];
            row[1 * N + j] = zj[j][1];
            row[2 * N + j] = zj[j][2];
            row[3 * N + j] = (real)0;
            row[4 * N + j] = (real)0;
            row[5 * N + j] = (real)0;
        }
    }
}

// Rows K0..K0+2 of a row-major 6 x N Jacobian row, column j seen as the 3-vector v[j][0..2] (the indexing of the
// register stash arrays): lets chain_forward write its stash straight into the Jacobian row in shared memory.
template <typename real, int N, int K0>
struct JRowCols {
    real *row;
    struct Col {
        real *p;
        __device__ __forceinline__ real &operator[](int i) const { return p[i * N]; }
    };
    __device__ __forceinline__ Col operator[](int j) const { return Col{row + K0 * N + j}; }
};

// The DH-like walk's stash written into the row itself (JRowCols<3> for z_j, JRowCols<0> for p_j): rows 3..5 already
// hold their final values z_j, rows 0..2 hold p_j and are overwritten with z_j x (p_e - p_j) -- the expressions of
// jacob0_row, so the result is bit-identical to the register form.
template <typename real, int N>
__device__ __forceinline__ void jacob0_from_stash(const Pose<real> &T, real *row)
{
#pragma unroll
    for (int j = 0; j < N; j++) {
        const real z0 = row[3 * N + j], z1 = row[4 * N + j], z2 = row[5 * N + j];
        const real dx = T.p[0] - row[0 * N + j], dy = T.p[1] - row[1 * N + j], dz = T.p[2] - row[2 * N + j];
        row[0 * N + j] = fma(z1, dz, -(z2 * dy));
        row[1 * N + j] = fma(z2, dx, -(z0 * dz));
        row[2 * N + j] = fma(z0, dy, -(z1 * dx));
    }
}

// ------------------------------------------------------------------ per-warp staging of output tiles
// A tile of 32 rows x ROW_ELEMS reals is staged in units of UB bytes (16 when a row is a whole
// number of 16-byte units, else 8) with a row stride of S units, S odd and >= units per row, so
// that the one-row-per-lane vector stores are bank-conflict free.  The warp then copies the tile
// to global memory unit by unit: consecutive lanes -> consecutive units -> full-width coalesced
// stores.  When S equals the units per row the stage is the exact image of the output block.
template <typename real, int ROW_ELEMS>
struct TileStage {
    static constexpr int ROW_BYTES = ROW_ELEMS * (int)sizeof(real);
    static constexpr int UB = (ROW_BYTES % 16 == 0) ? 16 : (ROW_BYTES % 8 == 0 ? 8 : 4);
    static constexpr int RU = ROW_BYTES / UB;          // units per row
    // bank-conflict degree of one-row-per-lane vector stores at row stride RU units
    static constexpr int cgcd(int a, int b) { return b ? cgcd(b, a % b) : a; }
    static constexpr int WAVE = UB == 16 ? 8 : (UB == 8 ? 16 : 32); // lanes served per shared-memory wavefront
    // exact image of the output block when that costs at most 2-way conflicts, else pad to an odd stride
    static constexpr int S = (cgcd(RU, WAVE) <= 2) ? RU : (RU | 1);
    static constexpr bool EXACT = (S == RU);
    static constexpr int BYTES = 32 * S * UB;
    typedef typename std::conditional<UB == 16, uint4, typename std::conditional<UB == 8, uint2, unsigned>::type>::type unit_t;

    // lane writes its row (ROW_ELEMS values in registers) with vector stores
    static __device__ __forceinline__ void put_row(unsigned char *stage, int lane, const real *row)
    {
        unit_t *dst = reinterpret_cast<unit_t *>(stage) + lane * S;
#pragma unroll
        for (int u = 0; u < RU; u++) {
            unit_t v;
            if constexpr (sizeof(real) == 8) {
                if constexpr (UB == 16) {
                    v.x = __double2loint(row[2 * u]); v.y = __double2hiint(row[2 * u]);
                    v.z = __double2loint(row[2 * u + 1]); v.w = __double2hiint(row[2 * u + 1]);
                } else {
                    v.x = __double2loint(row[u]); v.y = __double2hiint(row[u]);
                }
            } else {
                if constexpr (UB == 16) {
                    v.x = __float_as_int(row[4 * u]); v.y = __float_as_int(row[4 * u + 1]);
                    v.z = __float_as_int(row[4 * u + 2]); v.w = __float_as_int(row[4 * u + 3]);
                } else if constexpr (UB == 8) {
                    v.x = __float_as_int(row[2 * u]); v.y = __float_as_int(row[2 * u + 1]);
                } else {
                    v = (unsigned)__float_as_int(row[u]);
                }
            }
            dst[u] = v;
        }
    }

    // Asynchronous drain through the TMA engine (cp.async.bulk shared -> global): no LDS/STG
    // instructions, no registers, and the warp moves on to its next tile while the copy is in
    // flight.  Exact-image stages go out as ONE bulk copy issued by lane 0; padded stages as one
    // bulk copy per row issued by the lane that owns the row.  Returns false when this tile cannot
    // use bulk copies (size / alignment not a multiple of 16 bytes): caller falls back to drain().
    // Call wait_reads() before the stage is written again.
    static __device__ __forceinline__ bool drain_async(unsigned char *stage, real *gout, int rows_here, int lane)
    {
        if constexpr (EXACT) {
            const unsigned bytes = (unsigned)rows_here * ROW_BYTES;
            if ((bytes & 15u) || (reinterpret_cast<uintptr_t>(gout) & 15)) return false; // cp.async.bulk needs 16-byte size and address
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                const unsigned s = (unsigned)__cvta_generic_to_shared(stage);
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gout), "r"(s), "r"(bytes) : "memory");
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            return true;
        } else if constexpr (UB == 16) {
            if (reinterpret_cast<uintptr_t>(gout) & 15) return false;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane < rows_here) {
                const unsigned s = (unsigned)__cvta_generic_to_shared(stage + (size_t)lane * S * UB);
                const unsigned bytes = ROW_BYTES;
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gout + (size_t)lane * ROW_ELEMS), "r"(s), "r"(bytes) : "memory");
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            return true;
        } else {
            return false;
        }
    }
    // every lane's outstanding bulk copies have finished READING shared memory
    static __device__ __forceinline__ void wait_reads()
    {
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncwarp();
    }
    static __device__ __forceinline__ void wait_all()
    {
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }

    // warp copies the staged tile to gout (the tile's block of the output array)
    static __device__ __forceinline__ void drain(const unsigned char *stage, real *gout, int rows_here, int lane)
    {
        const unit_t *src = reinterpret_cast<const unit_t *>(stage);
        unit_t *dst = reinterpret_cast<unit_t *>(gout);
        constexpr int ITERS = RU; // 32 rows * RU units / 32 lanes
        if (rows_here == 32) {
            if constexpr (S == RU) { // exact image: flat copy, immediate offsets
#pragma unroll
                for (int it = 0; it < ITERS; it++) dst[it * 32 + lane] = src[it * 32 + lane];
            } else if constexpr (32 % RU == 0) { // whole rows per warp pass: immediate offsets again
                constexpr int RPP = 32 / RU; // rows per pass
                const int base = (lane / RU) * S + (lane % RU);
#pragma unroll
                for (int it = 0; it < ITERS; it++) dst[it * 32 + lane] = src[base + it * RPP * S];
            } else { // incremental (row, col) walk: no division in the loop
                int c = lane % RU;
                int off = (lane / RU) * S + c;
#pragma unroll
                for (int it = 0; it < ITERS; it++) {
                    dst[it * 32 + lane] = src[off];
                    c += 32 % RU;
                    off += (32 / RU) * S + (32 % RU);
                    if (c >= RU) { c -= RU; off += S - RU; }
                }
            }
        } else { // ragged last tile
            const int lim = rows_here * RU;
            for (int u = lane; u < lim; u += 32) {
                int r = u / RU, c = u - r * RU;
                dst[u] = src[r * S + c];
            }
        }
    }
};

// pose row: 16 reals, bottom row 0 0 0 1
template <typename real>
__device__ __forceinline__ void pose_to_row(const Pose<real> &T, real *row)
{
#pragma unroll
    for (int i = 0; i < 3; i++) {
        row[i * 4 + 0] = T.c0[i];
        row[i * 4 + 1] = T.c1[i];
        row[i * 4 + 2] = T.c2[i];
        row[i * 4 + 3] = T.p[i];
    }
    row[12] = (real)0; row[13] = (real)0; row[14] = (real)0; row[15] = (real)1;
}

// The pose block needs no transposition through shared memory: a row is 16 contiguous reals
// (128 B in fp64, 64 B in fp32), so each lane stores its own row with full-sector vector stores
// straight from registers.
template <typename real>
__device__ __forceinline__ void store_pose_row(const Pose<real> &T, real *grow)
{
    real row[16];
    pose_to_row(T, row);
    if constexpr (sizeof(real) == 8) {
        double4 *g = reinterpret_cast<double4 *>(grow);
#pragma unroll
        for (int u = 0; u < 4; u++) { // 256-bit stores (sm_100): one full 32-byte sector per instruction per lane
            asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(g + u), "d"(row[4 * u]), "d"(row[4 * u + 1]),
                         "d"(row[4 * u + 2]), "d"(row[4 * u + 3]) : "memory");
        }
    } else {
        float4 *g = reinterpret_cast<float4 *>(grow);
#pragma unroll
        for (int u = 0; u < 2; u++) {
            asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(g + 2 * u), "f"(row[8 * u]),
                         "f"(row[8 * u + 1]), "f"(row[8 * u + 2]), "f"(row[8 * u + 3]), "f"(row[8 * u + 4]),
                         "f"(row[8 * u + 5]), "f"(row[8 * u + 6]), "f"(row[8 * u + 7]) : "memory");
        }
    }
}

// ------------------------------------------------------------------ q tile loading
// qmode 1: the smem tile is the exact image of the 32 x ldq global block, filled with 16-byte
//          cp.async (no registers, asynchronous: used to prefetch the next tile);
// qmode 0: padded rows (stride ldq|1), element-wise copy -- used when the exact image would make
//          the one-row-per-lane reads collide (gcd(ldq, banks) > 2) or q is not 16-byte aligned.
__device__ __forceinline__ void cp_async16(void *smem, const void *gmem)
{
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

template <typename real>
__device__ __forceinline__ void load_q_tile(real *sq, const real *__restrict__ gq, int rows_here, int ldq,
                                            float inv_ldq, int qmode, int lane)
{
    const int cnt = rows_here * ldq;
    if (qmode == 1) {
        if (rows_here == 32) {
            const int units = (32 * ldq * (int)sizeof(real)) >> 4;
            const uint4 *g = reinterpret_cast<const uint4 *>(gq);
            uint4 *s = reinterpret_cast<uint4 *>(sq);
            for (int u = lane; u < units; u += 32) cp_async16(s + u, g + u);
        } else {
            for (int i = lane; i < cnt; i += 32) sq[i] = gq[i];
        }
    } else {
        const int ldqp = ldq | 1;
        for (int i = lane; i < cnt; i += 32) {
            int r = __float2int_rz(((float)i + 0.5f) * inv_ldq);
            int c = i - r * ldq;
            sq[r * ldqp + c] = gq[i];
        }
    }
}

// Under a saturated write stream a DRAM read waits far longer than one tile's worth of work
// (ncu: the warps' top stall was the cp.async wait, profiles/r01_fkj_v4.md), so the q block of a
// tile further ahead is pulled into L2 with fire-and-forget prefetches; the cp.async that later
// stages it into shared memory is then an L2 hit.  Costs one instruction, no registers, no smem.
template <typename real>
__device__ __forceinline__ void prefetch_q_tile_l2(const real *gq, int rows_here, int ldq, int lane)
{
    const char *p = reinterpret_cast<const char *>(gq);
    const char *first = reinterpret_cast<const char *>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)127);
    const char *end = p + (size_t)rows_here * ldq * sizeof(real);
    for (const char *a = first + (size_t)lane * 128; a < end; a += 32 * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
}

// Programmatic dependent launch: every fkj kernel is launched with programmatic stream serialization (fkj_launch_pdl),
// so it may become resident while the previous kernel on the stream is still draining.  griddepcontrol.wait blocks
// until that kernel has completed and its writes are visible (q may be what it wrote), so it precedes every global
// access; launch_dependents then lets the next fkj call be scheduled onto the SMs this grid frees.  Both are no-ops
// when the kernel was launched without the attribute.
__device__ __forceinline__ void pdl_wait_then_release()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// bytes of per-warp shared memory: [q tile][output stage]
template <typename real>
inline size_t fkj_q_bytes(int ldq) { return ((size_t)32 * (ldq | 1) * sizeof(real) + 15) & ~(size_t)15; }

template <typename real, int N>
inline size_t fkj_warp_smem(int ldq, bool wt, bool wj)
{
    (void)wt; // the pose block is stored straight from registers
    size_t j = wj ? (size_t)TileStage<real, 6 * N>::BYTES : 0;
    return fkj_q_bytes<real>(ldq) + j;
}

// registers: cap at 128/thread (4 resident blocks of 128 threads per SM) where the stash allows it
template <typename real, int N, bool WJ>
struct FkjBounds {
    static constexpr int MINB = (!WJ) ? (sizeof(real) == 4 ? 8 : 6) : (sizeof(real) == 4 ? 4 : (N <= 7 ? 4 : 3));
};

// ------------------------------------------------------------------ forward walk: pose and/or base-frame Jacobian
template <typename real, int N, bool WT, bool WJ, int PROF>
__global__ void __launch_bounds__(B2K_THREADS, FkjBounds<real, N, WJ>::MINB)
k_fkj_forward(const __grid_constant__ ChainP<real, N> P, const real *__restrict__ q, long long nrows, int ldq,
              float inv_ldq, int qmode, real *__restrict__ Tout, real *__restrict__ Jout, int warp_smem_bytes,
              int q_bytes, int tpw, int dbg)
{
    // dbg (measurement skeletons, b2k_set_variant 2 / 3): bit 0 = skip the chain walk (memory
    // traffic only), bit 1 = skip the output stores (arithmetic only).  0 in normal operation.
    pdl_wait_then_release();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    unsigned char *wbase = smem_raw + (size_t)warp * warp_smem_bytes;
    real *sq = reinterpret_cast<real *>(wbase);
    unsigned char *so = wbase + q_bytes;
    const int ldqs = qmode ? ldq : (ldq | 1);
    const long long ntiles = (nrows + 31) >> 5;
    // a warp owns `tpw` CONSECUTIVE tiles (one-shot grid: tpw small; persistent measurement variant: all of its share)
    const long long tstride = 1;
    long long tile = ((long long)blockIdx.x * B2K_WARPS_PER_BLOCK + warp) * tpw;
    const long long tile_end = (tile + tpw < ntiles) ? tile + tpw : ntiles;
    if (tile < tile_end) {
        const long long row0 = tile << 5;
        load_q_tile<real>(sq, q + row0 * ldq, (int)((nrows - row0) < 32 ? (nrows - row0) : 32), ldq, inv_ldq, qmode, lane);
#pragma unroll
        for (int k = 1; k < B2K_L2_PREFETCH_TILES; k++) {
            const long long ft = tile + k * tstride;
            if (ft < tile_end) {
                const long long r0 = ft << 5;
                prefetch_q_tile_l2<real>(q + r0 * ldq, (int)((nrows - r0) < 32 ? (nrows - r0) : 32), ldq, lane);
            }
        }
    }
    for (; tile < tile_end; tile += tstride) {
        const long long row0 = tile << 5;
        const int rows_here = (int)((nrows - row0) < 32 ? (nrows - row0) : 32);
        cp_async_wait_all();
        __syncwarp();
        const real *myq = sq + (lane < rows_here ? lane : 0) * ldqs;

        Pose<real> T;
        real zj[WJ ? N : 1][3], pj[WJ ? N : 1][3];
        real qrow[N];
#pragma unroll
        for (int j = 0; j < N; j++) qrow[j] = myq[P.jidx[j]];
        __syncwarp(); // every lane holds its q row in registers: prefetch the next tile's q now
        {
            const long long nt = tile + tstride;
            if (nt < tile_end) {
                const long long r0 = nt << 5;
                load_q_tile<real>(sq, q + r0 * ldq, (int)((nrows - r0) < 32 ? (nrows - r0) : 32), ldq, inv_ldq, qmode, lane);
            }
            const long long ft = tile + B2K_L2_PREFETCH_TILES * tstride;
            if (ft < tile_end) {
                const long long r0 = ft << 5;
                prefetch_q_tile_l2<real>(q + r0 * ldq, (int)((nrows - r0) < 32 ? (nrows - r0) : 32), ldq, lane);
            }
        }
        if (dbg & 1) { // memory skeleton: fabricate outputs from q without walking the chain
            pose_from_const(T, P.A[0]);
            T.p[0] = qrow[0];
            if (WJ) {
#pragma unroll
                for (int j = 0; j < N; j++)
#pragma unroll
                    for (int i = 0; i < 3; i++) { zj[j][i] = qrow[j]; pj[j][i] = qrow[(j + i) % N]; }
            }
        } else {
            chain_forward<real, N, WJ, PROF>(P, [&](int j, int) { return qrow[j]; }, T, zj, pj);
        }
        if (dbg & 2) { // arithmetic skeleton: keep the results alive without writing them
            real acc = T.p[0] + T.c0[0] + T.c1[1] + T.c2[2] + T.p[1] + T.p[2];
            if (WJ) {
#pragma unroll
                for (int j = 0; j < N; j++) acc += zj[j][0] * pj[j][1] + zj[j][1] * pj[j][2] + zj[j][2] * pj[j][0];
            }
            if (acc == (real)123456.789) Tout[row0] = acc;
            continue;
        }
        if (WT) {
            Pose<real> Tb = T;
            if (P.has_base) pose_mul_const_left(Tb, P.B, AK_GEN | AK_TX | AK_TY | AK_TZ);
            if (lane < rows_here) store_pose_row<real>(Tb, Tout + (row0 + lane) * 16);
        }
        if (WJ) {
            typedef TileStage<real, 6 * N> JS;
            real row[6 * N];
            jacob0_row<real, N, PROF>(P, T, zj, pj, row);
            JS::wait_reads(); // the previous tile's bulk copy has finished reading the stage
            JS::put_row(so, lane, row);
            if (!JS::drain_async(so, Jout + row0 * (6 * N), rows_here, lane)) {
                __syncwarp();
                JS::drain(so, Jout + row0 * (6 * N), rows_here, lane);
                __syncwarp();
            }
        }
    }
    cp_async_wait_all();
    if (WJ) TileStage<real, 6 * N>::wait_all();
}

// Backward walk of a DH-like chain (unflipped Rz joints, Rx-form inter-joint constants): U starts at the tail
// constant and is left-multiplied towards the base; column j of Je is read off U before joint j is applied
// (reference _ETS_jacobe, methods.cpp:219-316).  row = Je, row-major 6 x N.
template <typename real, int N>
__device__ __forceinline__ void backward_walk_dh(const ChainP<real, N> &P, const real *eta, Pose<real> &U, real *row)
{
    real sn[N], cs[N];
    b2k_sincos_batch<real, N>(eta, P.trig, sn, cs);
#pragma unroll
    for (int j = N - 1; j >= 0; j--) {
        real col[6];
        je_col_rev<real, 2>(U, (real)1, col);
#pragma unroll
        for (int k = 0; k < 6; k++) row[k * N + j] = col[k];
        rot_rows<real, 0, 1>(U, sn[j], cs[j]);
        if (j > 0) { // left-multiply by the Rx-form constant A_j
            const real *A = P.A[j];
            real *cols[4] = {U.c0, U.c1, U.c2, U.p};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                real a = cols[k][1], b = cols[k][2];
                cols[k][1] = fma(A[5], a, A[6] * b);
                cols[k][2] = fma(A[9], a, A[10] * b);
            }
            U.p[0] += A[3]; U.p[1] += A[7]; U.p[2] += A[11];
        } else {
            pose_mul_const_left(U, P.A[0], P.akind[0]);
        }
    }
}

// ------------------------------------------------------------------ forward walk, lean form for the common call
// k_fkj_forward above is general: any row stride / jindex permutation / alignment, ragged tiles, several tiles per
// warp, measurement skeletons.  ncu on the pose-only fp32 kernel (profiles/r01_fkine_f32.txt) showed what that
// generality costs on a one-shot grid, where every warp pays the prologue for a single tile: ~300 of 714 issued
// instructions per tile were integer / control (IMAD, ISETP, LOP3, BRA, BSSY ...), and the kernel was issue-bound.
// This kernel is the same walk with everything about the call fixed at compile time: DH-like chain (PROF 1),
// q rows exactly N wide with jindex j = column j, 16-byte aligned q, one FULL tile per warp.  The launcher uses it
// for the full tiles of such calls and hands a ragged tail (nrows % 32 rows) to the general kernel.
//
// Jacobian stash (SMEM_STASH).  Held in registers, the walk's z_j / p_j stash is 6N reals per lane: 84 of the 128
// registers of the fp64 Panda kernel, which capped it at 4 resident blocks (16 warps) per SM -- too few to cover a
// DRAM round trip under the saturated write stream.  So fp64 kernels keep the stash in the lane's own row of the
// J stage (exactly 6N reals): z_j is written to its final place in rows 3..5 as soon as it is known, p_j to the
// row 0..2 places as scratch, and jacob0_from_stash finishes the row in place.  The q tile is the front of that stage.
// The stash's shared accesses run at the row stride of 6N reals.  For odd N the compiler pairs consecutive joints into
// 16-byte accesses, which are conflict-free at that stride; for even N they would be 2-way (16 B) to 4-way (8 B)
// bank-conflicted.  So only odd N <= 7 take it (N = 7: 96 registers, 43,008 B per block, 5 blocks per SM), and only in
// the fused pose + Jacobian kernel: the Jacobian-only one spills 48 B when held to 96 registers.
template <typename real, int N>
struct FkjFast {
    static constexpr int QBYTES = 32 * N * (int)sizeof(real);          // multiple of 128
    static constexpr int QUNITS = QBYTES / 16;
    static constexpr bool SMEM_STASH = sizeof(real) == 8 && (N % 2) == 1 && N <= 7;
    static constexpr int WB_POSE = QBYTES;                                  // per-warp shared memory, pose only
    static constexpr int WB_JAC = QBYTES + TileStage<real, 6 * N>::BYTES;   // with the Jacobian stage after the q tile
    static constexpr int WB_JAC_SS = TileStage<real, 6 * N>::BYTES;         // q tile inside the Jacobian stage
    __host__ __device__ static constexpr bool stash(bool wt, bool wj) { return wt && wj && SMEM_STASH; }
    __host__ __device__ static constexpr int wb(bool wt, bool wj) { return !wj ? WB_POSE : (stash(wt, wj) ? WB_JAC_SS : WB_JAC); }
    __host__ __device__ static constexpr int minb(bool wt, bool wj)
    {
        return stash(wt, wj) ? 5 : (wj ? FkjBounds<real, N, true>::MINB : FkjBounds<real, N, false>::MINB);
    }
};

// A lean kernel's q tile: L2 prefetch of the tile `pf_ahead` tiles further on (the launcher passes one resident grid's
// worth, so that tile's warp starts about one warp lifetime later and finds its q in L2), then 16-byte cp.async of
// this tile into shared memory.  Returns after the tile has landed and is visible to the whole warp.
template <typename real, int N>
__device__ __forceinline__ void lean_load_q(const real *q, int tile, int ntiles, int pf_ahead, real *sq, int lane)
{
    typedef FkjFast<real, N> F;
    if (lane == 0 && tile < ntiles - pf_ahead) {
        const real *pf = q + (size_t)(tile + pf_ahead) * (32 * N);
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(pf), "r"((unsigned)F::QBYTES) : "memory");
    }
    const uint4 *g = reinterpret_cast<const uint4 *>(q + (size_t)tile * (32 * N));
    uint4 *sdst = reinterpret_cast<uint4 *>(sq);
#pragma unroll
    for (int u = 0; u < (F::QUNITS + 31) / 32; u++) {
        const int idx = u * 32 + lane;
        if (F::QUNITS % 32 == 0 || idx < F::QUNITS) cp_async16(sdst + idx, g + idx);
    }
    cp_async_wait_all();
    __syncwarp();
}

template <typename real, int N, bool WT, bool WJ>
__global__ void __launch_bounds__(B2K_THREADS, FkjFast<real, N>::minb(WT, WJ))
k_fkj_fast(const __grid_constant__ ChainP<real, N> P, const real *__restrict__ q, int ntiles, int pf_ahead,
           real *__restrict__ Tout, real *__restrict__ Jout)
{
    pdl_wait_then_release();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef FkjFast<real, N> F;
    typedef TileStage<real, 6 * N> JS;
    constexpr bool STASH = F::stash(WT, WJ);
    static_assert(!STASH || JS::EXACT, "the stash needs the stage to be the exact image of the J block");
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int tile = blockIdx.x * B2K_WARPS_PER_BLOCK + warp;
    if (tile >= ntiles) return;
    unsigned char *wbase = smem_raw + warp * F::wb(WT, WJ);
    real *sq = reinterpret_cast<real *>(wbase);
    lean_load_q<real, N>(q, tile, ntiles, pf_ahead, sq, lane);
    real qrow[N];
#pragma unroll
    for (int j = 0; j < N; j++) qrow[j] = sq[lane * N + j];
    unsigned char *so = wbase + (STASH ? 0 : F::QBYTES); // the J stage
    real *srow = reinterpret_cast<real *>(so) + lane * (6 * N); // this lane's row of it (stash form)
    Pose<real> T;
    if constexpr (STASH) {
        __syncwarp(); // the q tile is the front of the stage: every lane holds its q row before any lane overwrites it
        chain_forward<real, N, true, 1>(P, [&](int j, int) { return qrow[j]; }, T, JRowCols<real, N, 3>{srow},
                                        JRowCols<real, N, 0>{srow});
    }
    real zj[WJ && !STASH ? N : 1][3], pj[WJ && !STASH ? N : 1][3];
    if constexpr (!STASH) chain_forward<real, N, WJ, 1>(P, [&](int j, int) { return qrow[j]; }, T, zj, pj);
    const size_t row = (size_t)tile * 32 + lane;
    if (WT) {
        Pose<real> Tb = T;
        if (P.has_base) pose_mul_const_left(Tb, P.B, AK_GEN | AK_TX | AK_TY | AK_TZ);
        store_pose_row<real>(Tb, Tout + row * 16);
    }
    if (WJ) {
        if constexpr (STASH) {
            jacob0_from_stash<real, N>(T, srow);
        } else {
            real jrow[6 * N];
            jacob0_row<real, N, 1>(P, T, zj, pj, jrow);
            JS::put_row(so, lane, jrow);
        }
        real *gout = Jout + (size_t)tile * (32 * 6 * N);
        if (!JS::drain_async(so, gout, 32, lane)) {
            __syncwarp();
            JS::drain(so, gout, 32, lane);
        } else {
            JS::wait_all(); // the bulk copy reads this warp's shared memory: it must finish before the block may retire
        }
    }
}

// lean form of the backward walk (end-effector-frame Jacobian, optional pose): same contract as k_fkj_fast
template <typename real, int N, bool WT>
__global__ void __launch_bounds__(B2K_THREADS, FkjBounds<real, N, true>::MINB)
k_fkj_back_fast(const __grid_constant__ ChainP<real, N> P, const real *__restrict__ q, int ntiles, int pf_ahead,
                real *__restrict__ Tout, real *__restrict__ Jout)
{
    pdl_wait_then_release();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef FkjFast<real, N> F;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int tile = blockIdx.x * B2K_WARPS_PER_BLOCK + warp;
    if (tile >= ntiles) return;
    unsigned char *wbase = smem_raw + warp * F::WB_JAC;
    real *sq = reinterpret_cast<real *>(wbase);
    lean_load_q<real, N>(q, tile, ntiles, pf_ahead, sq, lane);
    real eta[N];
#pragma unroll
    for (int j = 0; j < N; j++) eta[j] = sq[lane * N + j];
    Pose<real> U;
    real jrow[6 * N];
    pose_from_const(U, P.A[N]);
    backward_walk_dh<real, N>(P, eta, U, jrow);
    if (WT) {
        Pose<real> Tb = U;
        if (P.has_base) pose_mul_const_left(Tb, P.B, AK_GEN | AK_TX | AK_TY | AK_TZ);
        store_pose_row<real>(Tb, Tout + ((size_t)tile * 32 + lane) * 16);
    }
    typedef TileStage<real, 6 * N> JS;
    unsigned char *so = wbase + F::QBYTES;
    JS::put_row(so, lane, jrow);
    real *gout = Jout + (size_t)tile * (32 * 6 * N);
    if (!JS::drain_async(so, gout, 32, lane)) {
        __syncwarp();
        JS::drain(so, gout, 32, lane);
    } else {
        JS::wait_all();
    }
}

// ------------------------------------------------------------------ backward walk: end-effector-frame Jacobian (+ pose)
// Reference _ETS_jacobe, methods.cpp:219-316: U starts at the tool and is left-multiplied by
// each ET walking from the tip to the base; column j is read off U before joint j is applied.
template <typename real, int N, bool WT, int PROF>
__global__ void __launch_bounds__(B2K_THREADS, FkjBounds<real, N, true>::MINB)
k_fkj_backward(const __grid_constant__ ChainP<real, N> P, const real *__restrict__ q, long long nrows, int ldq,
               float inv_ldq, int qmode, real *__restrict__ Tout, real *__restrict__ Jout, int warp_smem_bytes,
               int q_bytes, int tpw)
{
    pdl_wait_then_release();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    unsigned char *wbase = smem_raw + (size_t)warp * warp_smem_bytes;
    real *sq = reinterpret_cast<real *>(wbase);
    unsigned char *so = wbase + q_bytes;
    const int ldqs = qmode ? ldq : (ldq | 1);
    const long long ntiles = (nrows + 31) >> 5;
    // a warp owns `tpw` CONSECUTIVE tiles (one-shot grid: tpw small; persistent measurement variant: all of its share)
    const long long tstride = 1;
    long long tile = ((long long)blockIdx.x * B2K_WARPS_PER_BLOCK + warp) * tpw;
    const long long tile_end = (tile + tpw < ntiles) ? tile + tpw : ntiles;
    if (tile < tile_end) {
        const long long row0 = tile << 5;
        load_q_tile<real>(sq, q + row0 * ldq, (int)((nrows - row0) < 32 ? (nrows - row0) : 32), ldq, inv_ldq, qmode, lane);
    }
    for (; tile < tile_end; tile += tstride) {
        const long long row0 = tile << 5;
        const int rows_here = (int)((nrows - row0) < 32 ? (nrows - row0) : 32);
        cp_async_wait_all();
        __syncwarp();
        const real *myq = sq + (lane < rows_here ? lane : 0) * ldqs;

        Pose<real> U;
        real row[6 * N]; // Je, row-major 6 x N
        pose_from_const(U, P.A[N]);
        if constexpr (PROF == 1) { // DH-like chain: straight-line walk, batched sincos
            real eta[N];
#pragma unroll
            for (int j = 0; j < N; j++) eta[j] = myq[P.jidx[j]];
            backward_walk_dh<real, N>(P, eta, U, row);
        } else {
#pragma unroll
            for (int j = N - 1; j >= 0; j--) {
                const int ax = P.axis[j];
                const real sg = P.flip[j] ? (real)-1 : (real)1;
                real col[6];
                switch (ax) {
                case B2K_RX: je_col_rev<real, 0>(U, sg, col); break;
                case B2K_RY: je_col_rev<real, 1>(U, sg, col); break;
                case B2K_RZ: je_col_rev<real, 2>(U, sg, col); break;
                case B2K_TX: je_col_pri<real, 0>(U, sg, col); break;
                case B2K_TY: je_col_pri<real, 1>(U, sg, col); break;
                default: je_col_pri<real, 2>(U, sg, col); break;
                }
#pragma unroll
                for (int k = 0; k < 6; k++) row[k * N + j] = col[k];
                pose_joint_left(U, ax, sg * myq[P.jidx[j]], P.trig);
                pose_mul_const_left(U, P.A[j], P.akind[j]);
            }
        }
        __syncwarp();
        {
            const long long nt = tile + tstride;
            if (nt < tile_end) {
                const long long r0 = nt << 5;
                load_q_tile<real>(sq, q + r0 * ldq, (int)((nrows - r0) < 32 ? (nrows - r0) : 32), ldq, inv_ldq, qmode, lane);
            }
        }
        if (WT) {
            Pose<real> Tb = U;
            if (P.has_base) pose_mul_const_left(Tb, P.B, AK_GEN | AK_TX | AK_TY | AK_TZ);
            if (lane < rows_here) store_pose_row<real>(Tb, Tout + (row0 + lane) * 16);
        }
        {
            typedef TileStage<real, 6 * N> JS;
            JS::wait_reads();
            JS::put_row(so, lane, row);
            if (!JS::drain_async(so, Jout + row0 * (6 * N), rows_here, lane)) {
                __syncwarp();
                JS::drain(so, Jout + row0 * (6 * N), rows_here, lane);
                __syncwarp();
            }
        }
    }
    cp_async_wait_all();
    TileStage<real, 6 * N>::wait_all();
}

// ------------------------------------------------------------------ launcher
enum { FKJ_T = 1, FKJ_J0 = 2, FKJ_JE = 4 };

inline int b2k_gcd(int a, int b) { return b ? b2k_gcd(b, a % b) : a; }

// can the q tile be kept as an exact image in shared memory (16-byte cp.async path)?
template <typename real>
inline int fkj_qmode(const void *q, int ldq)
{
    if (((uintptr_t)q) & 15) return 0;
    const int slots = sizeof(real) == 8 ? 16 : 32; // distinct banks-worth of elements per wavefront
    return b2k_gcd(ldq, slots) <= 2 ? 1 : 0;
}

// Launches an fkj kernel with programmatic stream serialization (see pdl_wait_then_release): its blocks may become
// resident while the previous kernel on the stream drains, which hides the launch gap and the dispatch ramp between
// consecutive calls.  A runtime that rejects the attribute gets a plain launch.
template <typename... KArgs, typename... Args>
inline cudaError_t fkj_launch_pdl(void (*kern)(KArgs...), unsigned grid, size_t smem, cudaStream_t st, Args... args)
{
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(B2K_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, kern, args...) == cudaSuccess) return cudaSuccess;
    cudaGetLastError(); // clear the rejection
    kern<<<grid, B2K_THREADS, smem, st>>>(args...);
    return cudaGetLastError();
}

template <typename real, int N>
int fkj_launch_n(const b2k_chain_s *c, int mode, const real *q, long long nrows, int ldq, const double *base,
                 const double *tool, real *T, real *J, cudaStream_t st)
{
    ChainP<real, N> P;
    const bool wt = mode & FKJ_T, wj0 = mode & FKJ_J0, wje = mode & FKJ_JE;
    // pose-only: base folded into the first constant; fused: base applied to the pose at the end
    b2k_fill_chain<real, N>(c, base, tool, /*base_into_chain=*/(wt && !wj0 && !wje), P);
    const size_t qb = fkj_q_bytes<real>(ldq);
    const size_t wsm = (fkj_warp_smem<real, N>(ldq, wt, wj0 || wje) + 15) & ~(size_t)15;
    const size_t smem = wsm * B2K_WARPS_PER_BLOCK;
    const float inv_ldq = 1.0f / (float)ldq;
    if (wt && (((uintptr_t)T) & 31)) { b2k_set_error("fkj: T must be 32-byte aligned"); return B2K_ERR_INVALID; }
    if ((wj0 || wje) && (((uintptr_t)J) % TileStage<real, 6 * N>::UB)) {
        b2k_set_error("fkj: J must be %d-byte aligned", TileStage<real, 6 * N>::UB);
        return B2K_ERR_INVALID;
    }

    const int variant = b2k_get_variant();
    const int dbg = variant == 2 ? 1 : (variant == 3 ? 2 : 0);
    auto launch_impl = [&](auto kern, auto... extra) -> int {
        // (q, nrows, T, J are read here, at launch time: the lean path below may have advanced them to the ragged tail)
        const long long ntiles = (nrows + 31) / 32;
        const long long nblk_needed = (ntiles + B2K_WARPS_PER_BLOCK - 1) / B2K_WARPS_PER_BLOCK;
        const int qmode = fkj_qmode<real>(q, ldq);
        int per_sm = b2k_blocks_per_sm((const void *)kern, B2K_THREADS, smem);
        if (per_sm < 1) return per_sm < 0 ? per_sm : (b2k_set_error("fkj kernel does not fit on an SM (smem %zu B)", smem), B2K_ERR_INVALID);
        // One-shot grid, a few consecutive tiles per warp: the hardware block scheduler hands out
        // row ranges in address order as SMs free up, which keeps the set of DRAM pages being
        // written compact.  A persistent grid (variant 4) measured 15-20 % lower write bandwidth
        // on B200 (scripts/exp/exp_mem3.cu: 5.96 vs 6.73 TB/s for this exact store pattern).
        long long tpw = b2k_tiles_per_warp(wj0 || wje);
        if (variant == 4) { // persistent: as many blocks as fit, each warp a contiguous share of the tiles
            long long g = (long long)b2k_num_sms() * per_sm;
            if (g > nblk_needed) g = nblk_needed;
            tpw = (ntiles + g * B2K_WARPS_PER_BLOCK - 1) / (g * B2K_WARPS_PER_BLOCK);
        }
        long long grid = (ntiles + B2K_WARPS_PER_BLOCK * tpw - 1) / (B2K_WARPS_PER_BLOCK * tpw);
        if (grid < 1) grid = 1;
        if (grid > 0x7fffffffLL || tpw > 0x7fffffffLL) { b2k_set_error("fkj: batch too large for one launch"); return B2K_ERR_INVALID; }
        B2K_CUDA(fkj_launch_pdl(kern, (unsigned)grid, smem, st, P, q, nrows, ldq, inv_ldq, qmode, T, J, (int)wsm, (int)qb,
                                (int)tpw, extra...));
        b2k_count_launch();
        return B2K_OK;
    };
    auto launch = [&](auto kern) -> int { return launch_impl(kern, dbg); };   // forward kernels take dbg
    auto launch_b = [&](auto kern) -> int { return launch_impl(kern); };      // backward kernels do not

    // Lean kernel for the common call (see k_fkj_fast): full tiles there, a ragged tail through the general kernel.
    if (c->dh_like && c->dense_jindex && ldq == N && variant == 0 && !(((uintptr_t)q) & 15) && nrows >= 32 &&
        nrows / 32 <= 0x7fffffffLL / 2) {
        const int nfull = (int)(nrows / 32);
        auto launch_fast = [&](auto kern, size_t fsmem) -> int {
            int per_sm = b2k_blocks_per_sm((const void *)kern, B2K_THREADS, fsmem);
            if (per_sm < 1) return per_sm < 0 ? per_sm : (b2k_set_error("fkj fast kernel does not fit on an SM (smem %zu B)", fsmem), B2K_ERR_INVALID);
            const unsigned grid = (unsigned)((nfull + B2K_WARPS_PER_BLOCK - 1) / B2K_WARPS_PER_BLOCK);
            const int pf_ahead = b2k_num_sms() * per_sm * B2K_WARPS_PER_BLOCK; // one resident grid of tiles (lean_load_q)
            B2K_CUDA(fkj_launch_pdl(kern, grid, fsmem, st, P, q, nfull, pf_ahead, T, J));
            b2k_count_launch();
            return B2K_OK;
        };
        typedef FkjFast<real, N> F;
        int rc;
        if (wje) rc = wt ? launch_fast(k_fkj_back_fast<real, N, true>, (size_t)F::WB_JAC * B2K_WARPS_PER_BLOCK)
                         : launch_fast(k_fkj_back_fast<real, N, false>, (size_t)F::WB_JAC * B2K_WARPS_PER_BLOCK);
        else if (wt && wj0) rc = launch_fast(k_fkj_fast<real, N, true, true>, (size_t)F::wb(true, true) * B2K_WARPS_PER_BLOCK);
        else if (wt) rc = launch_fast(k_fkj_fast<real, N, true, false>, (size_t)F::WB_POSE * B2K_WARPS_PER_BLOCK);
        else rc = launch_fast(k_fkj_fast<real, N, false, true>, (size_t)F::WB_JAC * B2K_WARPS_PER_BLOCK);
        const long long done = (long long)nfull * 32;
        if (rc != B2K_OK || done == nrows) return rc;
        // ragged tail: the last nrows % 32 rows, general kernel on the slices that start at row `done`
        q += done * ldq;
        if (wt) T += done * 16;
        if (wj0 || wje) J += done * (6 * N);
        nrows -= done;
    }
    if (wje) {
        if (c->dh_like) return wt ? launch_b(k_fkj_backward<real, N, true, 1>) : launch_b(k_fkj_backward<real, N, false, 1>);
        return wt ? launch_b(k_fkj_backward<real, N, true, 0>) : launch_b(k_fkj_backward<real, N, false, 0>);
    }
    if (c->dh_like) {
        if (wt && wj0) return launch(k_fkj_forward<real, N, true, true, 1>);
        if (wt) return launch(k_fkj_forward<real, N, true, false, 1>);
        return launch(k_fkj_forward<real, N, false, true, 1>);
    }
    if (wt && wj0) return launch(k_fkj_forward<real, N, true, true, 0>);
    if (wt) return launch(k_fkj_forward<real, N, true, false, 0>);
    return launch(k_fkj_forward<real, N, false, true, 0>);
}

template <typename real>
int fkj_launch(const b2k_chain_s *c, int mode, const void *q, long long nrows, long long ldq, const double *base,
               const double *tool, void *T, void *J, cudaStream_t st)
{
#define B2K_CASE(NN) \
    case NN: return fkj_launch_n<real, NN>(c, mode, (const real *)q, nrows, (int)ldq, base, tool, (real *)T, (real *)J, st);
    switch (c->n) {
        B2K_CASE(1) B2K_CASE(2) B2K_CASE(3) B2K_CASE(4) B2K_CASE(5)
        B2K_CASE(6) B2K_CASE(7) B2K_CASE(8) B2K_CASE(9) B2K_CASE(10)
    default:
        b2k_set_error("fkj: unsupported joint count %d", c->n);
        return B2K_ERR_INVALID;
    }
#undef B2K_CASE
}
