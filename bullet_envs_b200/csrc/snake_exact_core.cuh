// snake_exact_core.cuh -- one environment per THREAD: the env-step with the motor rows eliminated.
//
// With the reference's motor settings (force = inf, snake.py:26-27; PyBullet default kd = 1) every
// motor row of the solver is the equality qd_j+ = kp (q*_j - q_j)/dt, so the 16 joints move on a
// prescribed trajectory and only the 6 rigid degrees of freedom of the whole chain remain unknown.
// The tick is then (oracle: tick_exact in oracle/snake_oracle.c, same rows, order, clamps, residual):
//   pass 1  tip-ward walk in world axes: kinematics, velocities, reference accelerations (base
//           acceleration zero, joint accelerations prescribed), Newton-Euler wrench of every body,
//           composite inertia of the frozen chain, cylinder-vs-plane contact geometry;
//   solve   the free rigid acceleration about the chain's centre of mass C (there the 6x6 composite
//           inertia is block diagonal: mass and a 3x3 rotational inertia);
//   rows    per contact: lever arm about C, effective masses, right-hand sides;
//   PGS     projected Gauss-Seidel on the rigid twist (6 numbers in registers): all normal rows, then
//           all friction pairs (implicit cone), <= 50 sweeps, Bullet's residual early exit;
//   pass 2  base-ward walk: inverse dynamics with the contact impulses -> applied motor torques
//           (getJointState()[3]), joint integration;
//   finish  base velocity/pose integration, joint-0 reaction force.
//
// Data placement (DESIGN.md section 5): the 13 base-state floats, the chain cursor and the solver's
// 6-vector live in registers; the contact-row table (32 contacts x 17 words, re-read by every sweep)
// lives in tensor memory or shared memory behind a row-storage policy (RowsT / RowsS below); joint
// angles/velocities/torques stay in the environment's 256 B record of the handle's [N][64] state
// array (L1 resident while a lane owns the environment); model tables are read from constant memory
// at warp-uniform addresses.
//
// The tick is WARP CONVERGENT (every lane executes every row-storage access; masked lanes commit
// nothing) because the tensor-memory accesses are warp-wide .sync.aligned instructions.
//
// Everything except RowsT is __host__ __device__ so that tests/hostemu can run the very same fp32
// code on the CPU (development check only; the product library contains the device code only).
#pragma once
#include "snake_step.cuh"

#ifdef __CUDACC__
#define SNK_HD __host__ __device__ __forceinline__
#else
#define SNK_HD inline
#endif

#define EB 32 // environments (= lanes) per warp

// unroll factors of the solver's row loops (normal rows / friction pairs)
#ifndef SNK_UNROLL_N
#define SNK_UNROLL_N 4
#endif
#ifndef SNK_UNROLL_F
#define SNK_UNROLL_F 2
#endif
// Operation orders of the solver rows (tools/screen_variants.py): the arithmetic is the same up to the association of the sums, but
// ptxas allocates registers differently for each, and every pair of source registers of one instruction that shares a register bank
// costs an issue cycle.  The defaults are the orders with the fewest conflicts in the SASS of the benchmarked kernel.
#ifndef SNK_VAR_G
#define SNK_VAR_G 1
#endif
#ifndef SNK_VAR_DW
#define SNK_VAR_DW 1
#endif
#ifndef SNK_VAR_F
#define SNK_VAR_F 0
#endif
#ifndef SNK_VAR_T
#define SNK_VAR_T 1
#endif
#ifndef SNK_VAR_U
#define SNK_VAR_U 1
#endif
#ifndef SNK_VAR_NDW
#define SNK_VAR_NDW 0
#endif
#define SNK_PRAGMA_(x) _Pragma(#x)
#define SNK_UNROLL(n) SNK_PRAGMA_(unroll n)

// Model tables for the exact kernel (fp32; constant memory on the device).
struct ExTables {
    float jR0[NJ][9];
    float jt[NJ][3];
    float jax[NJ][3];
    float jdamp[NJ];
    float mass[NB];
    float com[NB][3];
    float Ic[NB][6]; // xx xy xz yy yz zz about the COM, body axes
    float ccen[NC][3];
    float cax[NC][3];
    float cfr[NC][9];
    float crad[NC], ceh[NC] /* end * halflen */, cmar[NC], cbrk[NC];
    float hpt[NB][3];
    float fzax[3];
    float rootm, mtot, inv_mtot;
    int cstart[NB + 1]; // cylinders of body b are [cstart[b], cstart[b+1])
};

// -----------------------------------------------------------------------------------------------
// Contact-row storage.  One record of 17 words per contact and environment:
//   word  0      normal impulse                      (solver state)
//   words 1-2    lever arm r.x, r.y about the chain's centre of mass
//   word  3      invD_n                              (words 0-3 are all the normal sweep reads from the record)
//   word  4      r.z
//   words 5-9    friction directions d1.xyz, d2.x, d2.z (anisotropic, not normalised).  d2.y is not stored: the directions are
//                columns of the symmetric matrix A = Rl diag(aniso) Rl^T (d1 = -A e_y, d2 = A e_x), so d2.y = -d1.x
//   words 10-11  rhs_1 invD_1, rhs_2 invD_2
//   words 12-13  friction impulses                   (solver state)
//   words 14-15  invD_1, invD_2
//                (the impulses sit 2 words after rhs invD so that the two operands of  impulse + rhs invD  come from different
//                register banks when the 16 words arrive in 16 consecutive registers)
//   N1           rhs_n invD_n                        (only the normal sweep reads it)
// Words 0-15 live either in shared memory as [word/4][contact][lane] float4 columns (bank = lane) or in
// TENSOR MEMORY: TMEM lane = thread, column = 16 * contact + word, moved with tcgen05.ld/st 32x32b
// (sm_100a; the 512 columns of a warp's TMEM quadrant hold exactly 32 contacts x 16 words).  N1 is always in
// shared memory (4 KB per warp); the joint targets are in global memory (RowsS/RowsT::tg).
// -----------------------------------------------------------------------------------------------
struct RowsSmemStore {  // one warp, rows in shared memory: 69 632 B
    float4 X[4][NC][EB];
    float N1[NC][EB];
};
struct RowsTmemAux {    // one warp, rows in tensor memory: the shared-memory part, 4 096 B
    float N1[NC][EB];
};
typedef RowsSmemStore ExSmem;

// Both policies also carry `tg`, the 16 joint targets of the lane's current environment: a 64 B row of the handle's target
// scratch array in global memory (written when the lane takes the environment, L1/L2 resident while it owns it).
struct RowsS {
    static constexpr bool REGN = false; // invD_n / rhs_n invD_n come from the record, not from registers
    RowsSmemStore* s;
    int lane;
    float* tg;
    SNK_HD float& tgt(int j) const { return tg[j]; }
    SNK_HD void st_n1(int k, float a) const { s->N1[k][lane] = a; }
    SNK_HD void ld_n(int k, float4& x0, float& n1) const { x0 = s->X[0][k][lane]; n1 = s->N1[k][lane]; }
    SNK_HD void st16(int k, float4 x0, float4 x1, float4 x2, float4 x3) const {
        s->X[0][k][lane] = x0; s->X[1][k][lane] = x1; s->X[2][k][lane] = x2; s->X[3][k][lane] = x3;
    }
    SNK_HD void st12(int k, float4 x0, float4 x1, float4 x2) const { s->X[0][k][lane] = x0; s->X[1][k][lane] = x1; s->X[2][k][lane] = x2; }
    SNK_HD void ld16(int k, float4& x0, float4& x1, float4& x2, float4& x3) const {
        x0 = s->X[0][k][lane]; x1 = s->X[1][k][lane]; x2 = s->X[2][k][lane]; x3 = s->X[3][k][lane];
    }
    SNK_HD void st_ln(int k, float v) const { s->X[0][k][lane].x = v; }
    SNK_HD void st_lf(int k, float a, float b) const { *reinterpret_cast<float2*>(&s->X[3][k][lane].x) = make_float2(a, b); }
    SNK_HD void fence4(float4&) const {}
    SNK_HD void fence16(float4&, float4&, float4&, float4&) const {}
    SNK_HD void fence_st() const {}
    // storage-neutral names used by ex_tick (the hybrid policy RowsH stores the same words elsewhere)
    SNK_HD void st_tmp(int k, float4 t0, float4 t1, float4 t2) const { st12(k, t0, t1, t2); }
    SNK_HD void ld_tmp(int k, float4& t0, float4& t1, float4& t2) const { t0 = s->X[0][k][lane]; t1 = s->X[1][k][lane]; t2 = s->X[2][k][lane]; }
    SNK_HD void fence_tmp(float4&, float4&, float4&) const {}
    SNK_HD void st_rec(int k, float4 x0, float4 x1, float4 x2, float4 x3, float n1) const { st16(k, x0, x1, x2, x3); st_n1(k, n1); }
    SNK_HD void ld_regn(int, float&, float&) const {}
    SNK_HD void clr_lf(int) const {}
};

#ifdef __CUDACC__
// Rows in tensor memory.  Every access is a warp-wide .sync.aligned instruction: the code using this policy
// keeps the warp converged (inactive lanes compute on their stale record and are masked at the commits).
// Loads are asynchronous: the destination registers may only be read after fence4/fence16, which wait for
// the load AND tie the registers so that the compiler cannot move a use above the wait.
struct RowsT {
    static constexpr bool REGN = false;
    uint32_t taddr;  // TMEM address of this warp's quadrant: base + (32 * (warp % 4) << 16)
    RowsTmemAux* s;
    int lane;
    float* tg;
    __device__ __forceinline__ float& tgt(int j) const { return tg[j]; }
    __device__ __forceinline__ void st_n1(int k, float a) const { s->N1[k][lane] = a; }
    __device__ __forceinline__ void ld_n(int k, float4& x0, float& n1) const {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=f"(x0.x), "=f"(x0.y), "=f"(x0.z), "=f"(x0.w) : "r"(taddr + 16u * k) : "memory");
        n1 = s->N1[k][lane];
    }
    __device__ __forceinline__ void st4(uint32_t col, float4 v) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr + col), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
    }
    __device__ __forceinline__ void st16(int k, float4 x0, float4 x1, float4 x2, float4 x3) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr + 16u * k),
                     "f"(x0.x), "f"(x0.y), "f"(x0.z), "f"(x0.w), "f"(x1.x), "f"(x1.y), "f"(x1.z), "f"(x1.w), "f"(x2.x), "f"(x2.y), "f"(x2.z), "f"(x2.w),
                     "f"(x3.x), "f"(x3.y), "f"(x3.z), "f"(x3.w) : "memory");
    }
    __device__ __forceinline__ void st12(int k, float4 x0, float4 x1, float4 x2) const { st4(16u * k, x0); st4(16u * k + 4u, x1); st4(16u * k + 8u, x2); }
    __device__ __forceinline__ void ld16(int k, float4& x0, float4& x1, float4& x2, float4& x3) const {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                     : "=f"(x0.x), "=f"(x0.y), "=f"(x0.z), "=f"(x0.w), "=f"(x1.x), "=f"(x1.y), "=f"(x1.z), "=f"(x1.w), "=f"(x2.x), "=f"(x2.y), "=f"(x2.z),
                       "=f"(x2.w), "=f"(x3.x), "=f"(x3.y), "=f"(x3.z), "=f"(x3.w)
                     : "r"(taddr + 16u * k) : "memory");
    }
    __device__ __forceinline__ void st_ln(int k, float v) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr + 16u * k), "f"(v) : "memory");
    }
    __device__ __forceinline__ void st_lf(int k, float a, float b) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr + 16u * k + 12u), "f"(a), "f"(b) : "memory");
    }
    __device__ __forceinline__ void fence4(float4& x0) const {
        asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(x0.x), "+f"(x0.y), "+f"(x0.z), "+f"(x0.w)::"memory");
    }
    __device__ __forceinline__ void fence16(float4& x0, float4& x1, float4& x2, float4& x3) const {
        asm volatile("tcgen05.wait::ld.sync.aligned;"
                     : "+f"(x0.x), "+f"(x0.y), "+f"(x0.z), "+f"(x0.w), "+f"(x1.x), "+f"(x1.y), "+f"(x1.z), "+f"(x1.w), "+f"(x2.x), "+f"(x2.y), "+f"(x2.z),
                       "+f"(x2.w), "+f"(x3.x), "+f"(x3.y), "+f"(x3.z), "+f"(x3.w)::"memory");
    }
    __device__ __forceinline__ void fence_st() const { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
    __device__ __forceinline__ void st_tmp(int k, float4 t0, float4 t1, float4 t2) const { st12(k, t0, t1, t2); }
    __device__ __forceinline__ void ld_tmp(int k, float4& t0, float4& t1, float4& t2) const { float4 t3; ld16(k, t0, t1, t2, t3); }
    __device__ __forceinline__ void fence_tmp(float4& t0, float4& t1, float4& t2) const {
        asm volatile("tcgen05.wait::ld.sync.aligned;"
                     : "+f"(t0.x), "+f"(t0.y), "+f"(t0.z), "+f"(t0.w), "+f"(t1.x), "+f"(t1.y), "+f"(t1.z), "+f"(t1.w), "+f"(t2.x), "+f"(t2.y), "+f"(t2.z), "+f"(t2.w)::"memory");
    }
    __device__ __forceinline__ void st_rec(int k, float4 x0, float4 x1, float4 x2, float4 x3, float n1) const { st16(k, x0, x1, x2, x3); st_n1(k, n1); }
    __device__ __forceinline__ void ld_regn(int, float&, float&) const {}
    __device__ __forceinline__ void clr_lf(int) const {}
};

// HYBRID rows (the benchmarked kernel): every warp keeps 8 words of a record in tensor memory, 7 in shared memory and 2 in
// registers, so that EIGHT warps fit on an SM (two per scheduler; two per TMEM lane quadrant, 256 columns each):
//   tensor memory, column 8 k + w:  0 ln | 1 r.x | 2 r.y | 3 r.z | 4 la | 5 lb | 6 d1.x | 7 d1.y
//                                   (the normal sweep reads words 0-3 with one ld.x4, the friction sweep all 8 with one ld.x8;
//                                    the solver state ln / la, lb is written back with st.x1 / st.x2)
//   shared memory, per contact [A | B | C][lane]: A = (d1.z, d2.x, d2.z, rhs_1 invD_1)   B = (rhs_2 invD_2, invD_1)   C = invD_2   (28 KB per warp)
//   registers:                      invD_n and rhs_n invD_n of all 32 contacts (64 registers; only the normal sweep reads them, so only
//                                   that loop is fully unrolled).  The rows phase, whose contact index is dynamic, parks the two values
//                                   in the la / lb words (which start at zero); ld_regn / clr_lf move them into the registers and zero
//                                   the words in an unrolled prologue of the solver.
struct RowsHybStore { // 896 B per contact: the three loads of a record differ by constant offsets from one running address
    struct { float4 A[EB]; float2 B[EB]; float C[EB]; } c[NC];
};
struct RowsH {
    static constexpr bool REGN = true;
    uint32_t taddr;  // TMEM address of this warp's 256 columns: base + (32 * (warp % 4) << 16) + 256 * (warp / 4)
    RowsHybStore* s;
    int lane;
    float* tg;
    __device__ __forceinline__ float& tgt(int j) const { return tg[j]; }
    __device__ __forceinline__ void st8(uint32_t col, float a, float b, float c, float d, float e, float f, float g, float h) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr + col), "f"(a), "f"(b), "f"(c), "f"(d),
                     "f"(e), "f"(f), "f"(g), "f"(h) : "memory");
    }
    __device__ __forceinline__ void ld8(uint32_t col, float& a, float& b, float& c, float& d, float& e, float& f, float& g, float& h) const {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=f"(a), "=f"(b), "=f"(c), "=f"(d), "=f"(e), "=f"(f), "=f"(g), "=f"(h) : "r"(taddr + col) : "memory");
    }
    // pass-1 temporaries: t0, t1 in tensor memory, t2 in shared memory
    __device__ __forceinline__ void st_tmp(int k, float4 t0, float4 t1, float4 t2) const {
        st8(8u * k, t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w);
        s->c[k].A[lane] = t2;
    }
    __device__ __forceinline__ void ld_tmp(int k, float4& t0, float4& t1, float4& t2) const {
        ld8(8u * k, t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w);
        t2 = s->c[k].A[lane];
    }
    __device__ __forceinline__ void fence_tmp(float4& t0, float4& t1, float4&) const {
        asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(t0.x), "+f"(t0.y), "+f"(t0.z), "+f"(t0.w), "+f"(t1.x), "+f"(t1.y), "+f"(t1.z), "+f"(t1.w)::"memory");
    }
    // final record (logical layout of the other policies: x0 = ln rx ry invD_n | x1 = rz d1 | x2 = d2x d2z b1 b2 | x3 = la lb invD_1 invD_2)
    __device__ __forceinline__ void st_rec(int k, float4 x0, float4 x1, float4 x2, float4 x3, float n1) const {
        st8(8u * k, x0.x, x0.y, x0.z, x1.x, x0.w /* invD_n, parked */, n1 /* parked */, x1.y, x1.z);
        s->c[k].A[lane] = make_float4(x1.w, x2.x, x2.y, x2.z);
        s->c[k].B[lane] = make_float2(x2.w, x3.z);
        s->c[k].C[lane] = x3.w;
    }
    __device__ __forceinline__ void ld_regn(int k, float& idn, float& n1) const {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=f"(idn), "=f"(n1) : "r"(taddr + 8u * k + 4u) : "memory");
    }
    __device__ __forceinline__ void clr_lf(int k) const { st_lf(k, 0.f, 0.f); }
    __device__ __forceinline__ void ld_n(int k, float4& x0, float&) const { // (ln, rx, ry, rz)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=f"(x0.x), "=f"(x0.y), "=f"(x0.z), "=f"(x0.w) : "r"(taddr + 8u * k) : "memory");
    }
    __device__ __forceinline__ void ld16(int k, float4& x0, float4& x1, float4& x2, float4& x3) const {
        ld8(8u * k, x0.x, x0.y, x0.z, x1.x, x3.x, x3.y, x1.y, x1.z);
        const float4 a = s->c[k].A[lane];
        const float2 b = s->c[k].B[lane];
        x3.w = s->c[k].C[lane];
        x1.w = a.x; x2.x = a.y; x2.y = a.z; x2.z = a.w; x2.w = b.x; x3.z = b.y;
        x0.w = 0.f; // invD_n is not part of the friction record
    }
    __device__ __forceinline__ void st_ln(int k, float v) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr + 8u * k), "f"(v) : "memory");
    }
    __device__ __forceinline__ void st_lf(int k, float a, float b) const {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr + 8u * k + 4u), "f"(a), "f"(b) : "memory");
    }
    __device__ __forceinline__ void fence4(float4& x0) const {
        asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(x0.x), "+f"(x0.y), "+f"(x0.z), "+f"(x0.w)::"memory");
    }
    __device__ __forceinline__ void fence16(float4& x0, float4& x1, float4&, float4& x3) const { // the 8 words that come from tensor memory
        asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(x0.x), "+f"(x0.y), "+f"(x0.z), "+f"(x1.x), "+f"(x3.x), "+f"(x3.y), "+f"(x1.y), "+f"(x1.z)::"memory");
    }
    __device__ __forceinline__ void fence_regn8(float* a, float* b) const { // 8 contacts' worth of ld_regn destinations
        asm volatile("tcgen05.wait::ld.sync.aligned;"
                     : "+f"(a[0]), "+f"(a[1]), "+f"(a[2]), "+f"(a[3]), "+f"(a[4]), "+f"(a[5]), "+f"(a[6]), "+f"(a[7]), "+f"(b[0]), "+f"(b[1]), "+f"(b[2]),
                       "+f"(b[3]), "+f"(b[4]), "+f"(b[5]), "+f"(b[6]), "+f"(b[7])::"memory");
    }
    __device__ __forceinline__ void fence_st() const { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
};
#endif

// ---- small float3 helpers -------------------------------------------------------------------
struct V3 { float x, y, z; };
SNK_HD V3 mk(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
SNK_HD V3 operator+(V3 a, V3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
SNK_HD V3 operator-(V3 a, V3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
SNK_HD V3 operator*(V3 a, float s) { return mk(a.x * s, a.y * s, a.z * s); }
SNK_HD V3 cross(V3 a, V3 b) { return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
SNK_HD float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
SNK_HD V3 ld3(const float* p) { return mk(p[0], p[1], p[2]); }
struct M3 { float m[9]; }; // row-major
SNK_HD V3 mul(const M3& R, V3 v) {
    return mk(R.m[0] * v.x + R.m[1] * v.y + R.m[2] * v.z, R.m[3] * v.x + R.m[4] * v.y + R.m[5] * v.z, R.m[6] * v.x + R.m[7] * v.y + R.m[8] * v.z);
}
SNK_HD V3 mulT(const M3& R, V3 v) {
    return mk(R.m[0] * v.x + R.m[3] * v.y + R.m[6] * v.z, R.m[1] * v.x + R.m[4] * v.y + R.m[7] * v.z, R.m[2] * v.x + R.m[5] * v.y + R.m[8] * v.z);
}
SNK_HD M3 mul(const M3& A, const M3& B) {
    M3 o;
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) o.m[3 * i + j] = A.m[3 * i] * B.m[j] + A.m[3 * i + 1] * B.m[3 + j] + A.m[3 * i + 2] * B.m[6 + j];
    return o;
}
SNK_HD M3 mulBT(const M3& A, const M3& B) { // A B^T
    M3 o;
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) o.m[3 * i + j] = A.m[3 * i] * B.m[3 * j] + A.m[3 * i + 1] * B.m[3 * j + 1] + A.m[3 * i + 2] * B.m[3 * j + 2];
    return o;
}
// c + a1 b1 + a2 b2 + a3 b3 as three chained fmas, innermost term selected by ORDER (0: term 1 innermost, 1: term 3, 2: term 3 then 1)
template <int ORDER>
SNK_HD float ex_sum3(float a1, float b1, float a2, float b2, float a3, float b3, float c) {
    if (ORDER == 0) return fmaf(a3, b3, fmaf(a2, b2, fmaf(a1, b1, c)));
    if (ORDER == 1) return fmaf(a1, b1, fmaf(a2, b2, fmaf(a3, b3, c)));
    return fmaf(a2, b2, fmaf(a1, b1, fmaf(a3, b3, c)));
}
// a1 b1 + a2 b2 + a3 b3: a product and two fmas, the plain product selected by ORDER (0: term 3, 1: term 1, 2: term 3 with 1 and 2 swapped)
template <int ORDER>
SNK_HD float ex_dot3(float a1, float b1, float a2, float b2, float a3, float b3) {
    if (ORDER == 0) return fmaf(a1, b1, fmaf(a2, b2, a3 * b3));
    if (ORDER == 1) return fmaf(a3, b3, fmaf(a2, b2, a1 * b1));
    return fmaf(a2, b2, fmaf(a1, b1, a3 * b3));
}
struct S3 { float xx, xy, xz, yy, yz, zz; }; // symmetric 3x3
SNK_HD V3 mul(const S3& S, V3 v) {
    return mk(S.xx * v.x + S.xy * v.y + S.xz * v.z, S.xy * v.x + S.yy * v.y + S.yz * v.z, S.xz * v.x + S.yz * v.y + S.zz * v.z);
}
SNK_HD float ex_rcp(float x) {
#ifdef __CUDA_ARCH__
    return __frcp_rn(x);
#else
    return 1.0f / x;
#endif
}
// clamp to [-m, m] with the oracle's comparisons (a NaN passes through, unlike fminf/fmaxf)
SNK_HD float ex_clamp(float x, float m) { x = (x > m) ? m : x; return (x < -m) ? -m : x; }
// single MUFU.RSQ (flush-to-zero, no denormal fix-up): only used on the solver's serial chain
SNK_HD float ex_rsqrt_fast(float x) {
#ifdef __CUDA_ARCH__
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
#else
    return 1.0f / sqrtf(x);
#endif
}
// true when the predicate holds in every lane of the warp (the host emulation runs one environment at a time)
SNK_HD bool ex_all(bool p) {
#ifdef __CUDA_ARCH__
    return __all_sync(0xffffffffu, p);
#else
    return p;
#endif
}
SNK_HD int ex_popc(unsigned x) {
#ifdef __CUDA_ARCH__
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}
SNK_HD float ex_rsqrt(float x) {
#ifdef __CUDA_ARCH__
    return rsqrtf(x);
#else
    return 1.0f / sqrtf(x);
#endif
}
SNK_HD void ex_sincos(float a, float* s, float* c) {
#ifdef __CUDA_ARCH__
    sincosf(a, s, c);
#else
    *s = sinf(a); *c = cosf(a);
#endif
}
SNK_HD M3 quat_to_m3(const float* q) { // xyzw
    float x = q[0], y = q[1], z = q[2], w = q[3];
    M3 R;
    R.m[0] = 1 - 2 * (y * y + z * z); R.m[1] = 2 * (x * y - z * w);     R.m[2] = 2 * (x * z + y * w);
    R.m[3] = 2 * (x * y + z * w);     R.m[4] = 1 - 2 * (x * x + z * z); R.m[5] = 2 * (y * z - x * w);
    R.m[6] = 2 * (x * z - y * w);     R.m[7] = 2 * (y * z + x * w);     R.m[8] = 1 - 2 * (x * x + y * y);
    return R;
}
// child->parent rotation of joint j at angle q: jR0 * Rot(jax, q)
SNK_HD M3 joint_rot(const ExTables& T, int j, float q) {
    float s, c;
    ex_sincos(q, &s, &c);
    const float ax = T.jax[j][0], ay = T.jax[j][1], az = T.jax[j][2], C = 1.f - c;
    M3 Rq, R0;
    Rq.m[0] = c + ax * ax * C;      Rq.m[1] = ax * ay * C - az * s; Rq.m[2] = ax * az * C + ay * s;
    Rq.m[3] = ay * ax * C + az * s; Rq.m[4] = c + ay * ay * C;      Rq.m[5] = ay * az * C - ax * s;
    Rq.m[6] = az * ax * C - ay * s; Rq.m[7] = az * ay * C + ax * s; Rq.m[8] = c + az * az * C;
#pragma unroll
    for (int k = 0; k < 9; k++) R0.m[k] = T.jR0[j][k];
    return mul(R0, Rq);
}
// world inertia R Ic R^T of body b
SNK_HD S3 world_inertia(const ExTables& T, int b, const M3& R) {
    const float* I = T.Ic[b];
    M3 t; // R * Ic
#pragma unroll
    for (int i = 0; i < 3; i++) {
        float r0 = R.m[3 * i], r1 = R.m[3 * i + 1], r2 = R.m[3 * i + 2];
        t.m[3 * i] = r0 * I[0] + r1 * I[1] + r2 * I[2];
        t.m[3 * i + 1] = r0 * I[1] + r1 * I[3] + r2 * I[4];
        t.m[3 * i + 2] = r0 * I[2] + r1 * I[4] + r2 * I[5];
    }
    S3 S;
    S.xx = t.m[0] * R.m[0] + t.m[1] * R.m[1] + t.m[2] * R.m[2];
    S.xy = t.m[0] * R.m[3] + t.m[1] * R.m[4] + t.m[2] * R.m[5];
    S.xz = t.m[0] * R.m[6] + t.m[1] * R.m[7] + t.m[2] * R.m[8];
    S.yy = t.m[3] * R.m[3] + t.m[4] * R.m[4] + t.m[5] * R.m[5];
    S.yz = t.m[3] * R.m[6] + t.m[4] * R.m[7] + t.m[5] * R.m[8];
    S.zz = t.m[6] * R.m[6] + t.m[7] * R.m[7] + t.m[8] * R.m[8];
    return S;
}

// Per-thread view of the environment: registers (base state) + where its columns live.
struct ExEnv {
    float pos[3], quat[4], vel[3], omg[3]; // base state (SNK_S_POS..SNK_S_OMEGA), registers
    float* st;                             // &state[env][0]; slot k at st[k] (256 B record, L1 resident during the step)
    int tid;                               // column in the CTA's shared arrays
};
SNK_HD float& slot(const ExEnv& e, int k) { return e.st[k]; }

// Newton-Euler wrench of body b (force F, moment N about the COM) for COM acceleration ac, angular
// velocity w / acceleration al; gravity and Bullet's velocity damping (per merged body, D2) are the
// external forces.  vc = COM velocity.
SNK_HD void body_wrench(const ExTables& T, const KParams& P, int b, const S3& Iw, V3 w, V3 al, V3 vc, V3 ac, V3* F, V3* N) {
    const float m = T.mass[b];
    const float nv = sqrtf(dot(vc, vc)), nw = sqrtf(dot(w, w));
    const float kl = P.kl + P.kl * nv, ka = P.ka + P.ka * nw;
    V3 Iww = mul(Iw, w);
    *F = mk(m * (ac.x - P.g[0] + vc.x * kl), m * (ac.y - P.g[1] + vc.y * kl), m * (ac.z - P.g[2] + vc.z * kl));
    V3 t = cross(w, Iww), Ial = mul(Iw, al);
    *N = mk(Ial.x + t.x + Iww.x * ka, Ial.y + t.y + Iww.y * ka, Ial.z + t.z + Iww.z * ka);
}

// chain cursor: frame of the current body (position relative to the base origin) and its motion
struct ExCursor {
    M3 R;
    V3 p, w, v, al, acc; // al/acc: reference accelerations (zero base acceleration)
};

struct ExTickOut { int iterations; int contacts; float height; float err2_next; };

// Phase clocks (build variant -DSNK_PHASE_CLOCKS; tools/bench_phases.py reads them through snk_phase_clocks): lane 0 of every warp
// adds the clock64() cycles the warp spends in each phase of ex_tick -- 0 pass 1, 1 rows + solver prologue, 2 solver, 3 pass 2 +
// finish -- to row (global warp % SNK_CLK_WARPS) of snk_phase_clk.  The default build contains none of this.
#if defined(SNK_PHASE_CLOCKS) && defined(__CUDACC__)
#define SNK_CLK_WARPS 4096
#define SNK_CLK_PHASES 4
__device__ unsigned long long snk_phase_clk[SNK_CLK_WARPS][SNK_CLK_PHASES];
#endif
#if defined(SNK_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
struct ExPhaseClock {
    long long t = clock64();
    __device__ __forceinline__ void mark(int phase) {
        const long long now = clock64();
        if ((threadIdx.x & 31) == 0)
            atomicAdd(&snk_phase_clk[((blockIdx.x * blockDim.x + threadIdx.x) >> 5) % SNK_CLK_WARPS][phase], (unsigned long long)(now - t));
        t = now;
    }
};
#define SNK_PHASE_START ExPhaseClock phase_clock;
#define SNK_PHASE_MARK(k) phase_clock.mark(k);
#else
#define SNK_PHASE_START
#define SNK_PHASE_MARK(k)
#endif

// -----------------------------------------------------------------------------------------------
// One physics tick.  Returns the mean checkSnakeHeight z of the state at the START of the tick in
// out->height; when that height already exceeds the threshold and `abort_on_height` is set, nothing is
// modified and *aborted = true.  The function is WARP CONVERGENT: every lane executes every row-storage
// access; a lane with `active` false (no environment, or one that needs no tick) and an aborted lane run
// the arithmetic on whatever their registers hold and are masked at every commit.
// -----------------------------------------------------------------------------------------------
template <bool CONE, class Rows>
SNK_HD void ex_tick(const ExTables& T, const KParams& P, const Rows& R, ExEnv& e, bool active, bool abort_on_height, bool* aborted, ExTickOut* out) {
    const float dt = P.dt, inv_dt = P.inv_dt;
    const float p0z = e.pos[2];
    SNK_PHASE_START
    // ------------------------------------------------------------------ pass 1: tip-ward
    ExCursor c;
    c.R = quat_to_m3(e.quat);
    c.p = mk(0.f, 0.f, 0.f);
    c.w = ld3(e.omg); c.v = ld3(e.vel);
    c.al = mk(0.f, 0.f, 0.f); c.acc = mk(0.f, 0.f, 0.f);
    V3 wJ = mk(0.f, 0.f, 0.f), vJ = mk(0.f, 0.f, 0.f); // motion due to the NEW joint rates alone
    V3 h = mk(0.f, 0.f, 0.f), F0 = h, N0 = h;
    S3 J; J.xx = J.xy = J.xz = J.yy = J.yz = J.zz = 0.f;
    float hsum = 0.f, err2n = 0.f;
    unsigned act = 0u;
    // what pass 2 needs of body i >= 1, kept by pass 1 in six float4 (local memory): (Iw.xx xy xz yy | Iw.yz zz, a.x a.y | a.z, p |
    // cc, F.x | F.y F.z, N.x N.y | N.z) with a the world axis of joint i-1, p the frame origin and F, N the reference wrench of body i
    float4 keep[NJ][6];
    V3 ja = mk(0.f, 0.f, 0.f);
    float qn = slot(e, SNK_S_Q), qdn = slot(e, SNK_S_QD); // prefetched joint 0
#pragma unroll 1
    for (int i = 0; i < NB; i++) {
        if (i > 0) {
            const int j = i - 1;
            const float q = qn, qd = qdn, tg = R.tgt(j);
            if (i < NJ) { qn = slot(e, SNK_S_Q + i); qdn = slot(e, SNK_S_QD + i); }
            float qds = P.kp * (tg - q) * inv_dt;
            qds = ex_clamp(qds, P.maxvel);
            const float qdd = (qds - qd) * inv_dt;
            const float en = tg - (q + dt * qds);
            err2n += en * en;
            V3 d = mul(c.R, ld3(T.jt[j]));
            V3 wxd = cross(c.w, d);
            c.acc = c.acc + cross(c.al, d) + cross(c.w, wxd);
            c.v = c.v + wxd;
            vJ = vJ + cross(wJ, d);
            c.p = c.p + d;
            c.R = mul(c.R, joint_rot(T, j, q));
            const V3 a = mul(c.R, ld3(T.jax[j]));
            V3 wq = a * qd;
            c.al = c.al + a * qdd + cross(c.w, wq);
            c.w = c.w + wq;
            wJ = wJ + a * qds;
            ja = a;
        }
        // ---- body i
        {
            const float m = T.mass[i];
            V3 rc = mul(c.R, ld3(T.com[i]));
            V3 cc = c.p + rc;
            S3 Iw = world_inertia(T, i, c.R);
            V3 wxr = cross(c.w, rc);
            V3 vc = c.v + wxr;
            V3 ac = c.acc + cross(c.al, rc) + cross(c.w, wxr);
            V3 F, N;
            body_wrench(T, P, i, Iw, c.w, c.al, vc, ac, &F, &N);
            F0 = F0 + F;
            N0 = N0 + cross(cc, F) + N;
            h = h + cc * m;
            const float c2 = dot(cc, cc);
            J.xx += Iw.xx + m * (c2 - cc.x * cc.x); J.yy += Iw.yy + m * (c2 - cc.y * cc.y); J.zz += Iw.zz + m * (c2 - cc.z * cc.z);
            J.xy += Iw.xy - m * cc.x * cc.y; J.xz += Iw.xz - m * cc.x * cc.z; J.yz += Iw.yz - m * cc.y * cc.z;
            hsum += p0z + c.p.z + c.R.m[6] * T.hpt[i][0] + c.R.m[7] * T.hpt[i][1] + c.R.m[8] * T.hpt[i][2];
            if (i > 0) {
                float4* k = keep[i - 1];
                k[0] = make_float4(Iw.xx, Iw.xy, Iw.xz, Iw.yy); k[1] = make_float4(Iw.yz, Iw.zz, ja.x, ja.y);
                k[2] = make_float4(ja.z, c.p.x, c.p.y, c.p.z); k[3] = make_float4(cc.x, cc.y, cc.z, F.x);
                k[4] = make_float4(F.y, F.z, N.x, N.y);       k[5] = make_float4(N.z, 0.f, 0.f, 0.f);
            }
        }
        // ---- contacts of body i (A.5 with deviation D1: lowest point of the extreme rim)
#pragma unroll 1
        for (int k = T.cstart[i]; k < T.cstart[i + 1]; k++) {
            V3 axw = mul(c.R, ld3(T.cax[k]));
            V3 ce = c.p + mul(c.R, ld3(T.ccen[k])) + axw * T.ceh[k];
            const float az = axw.z;
            const float inv = ex_rsqrt(fmaxf(1.f - az * az, 1e-12f));
            V3 pc = ce + mk(az * axw.x * inv, az * axw.y * inv, (az * az - 1.f) * inv) * T.crad[k];
            const float dist = pc.z + p0z - T.cmar[k];
            act |= (dist < T.cbrk[k]) ? (1u << k) : 0u; // a separated contact gets an all-zero record below
            pc.z = dist - p0z; // contact point at height `dist` (world), relative to the base origin
            M3 cf, Rl;
#pragma unroll
            for (int q9 = 0; q9 < 9; q9++) cf.m[q9] = T.cfr[k][q9];
            Rl = mul(c.R, cf);
            // anisotropic friction directions: Rl diag(aniso) Rl^T t, t1 = (0,-1,0), t2 = (1,0,0)
            V3 l1 = mk(-Rl.m[3] * P.aniso[0], -Rl.m[4] * P.aniso[1], -Rl.m[5] * P.aniso[2]);
            V3 l2 = mk(Rl.m[0] * P.aniso[0], Rl.m[1] * P.aniso[1], Rl.m[2] * P.aniso[2]);
            V3 d1 = mul(Rl, l1), d2 = mul(Rl, l2);
            V3 uJ = vJ + cross(wJ, pc - c.p);
            // pass-1 temporaries in the record: (uJ.x | pc), (d1 | d2.x), (d2.y d2.z | uJ.y uJ.z)
            R.st_tmp(k, make_float4(uJ.x, pc.x, pc.y, pc.z), make_float4(d1.x, d1.y, d1.z, d2.x), make_float4(d2.y, d2.z, uJ.y, uJ.z));
        }
    }
    R.fence_st();
    out->height = hsum * (1.f / NB);
    out->err2_next = err2n;
    *aborted = abort_on_height && out->height > P.hthr;
    const bool commit = active && !*aborted;
    SNK_PHASE_MARK(0)

    // ------------------------------------------------------------------ free rigid motion about C
    const float invM = T.inv_mtot, M = T.mtot;
    const V3 hc = h * invM; // C - p0
    {
        const float h2 = dot(hc, hc);
        J.xx -= M * (h2 - hc.x * hc.x); J.yy -= M * (h2 - hc.y * hc.y); J.zz -= M * (h2 - hc.z * hc.z);
        J.xy += M * hc.x * hc.y; J.xz += M * hc.x * hc.z; J.yz += M * hc.y * hc.z;
    }
    S3 Ji; // J^-1 (adjugate)
    {
        const float c00 = J.yy * J.zz - J.yz * J.yz, c01 = J.xz * J.yz - J.xy * J.zz, c02 = J.xy * J.yz - J.xz * J.yy;
        const float det = J.xx * c00 + J.xy * c01 + J.xz * c02;
        const float id = 1.f / det;
        Ji.xx = c00 * id; Ji.xy = c01 * id; Ji.xz = c02 * id;
        Ji.yy = (J.xx * J.zz - J.xz * J.xz) * id; Ji.yz = (J.xy * J.xz - J.xx * J.yz) * id; Ji.zz = (J.xx * J.yy - J.xy * J.xy) * id;
    }
    const V3 NC0 = N0 - cross(hc, F0);
    const V3 alf = mul(Ji, NC0) * -1.f; // free angular acceleration
    const V3 aC = F0 * -invM;           // free acceleration of the point C
    const V3 w0 = ld3(e.omg), v0 = ld3(e.vel);
    V3 wf = w0 + alf * dt;                           // free angular velocity
    const V3 VC = v0 + cross(w0, hc) + aC * dt;      // free velocity of C (rigid field of the base)
    // (the base origin moves with this rigid field: v0' = VC - wf x hc, i.e. a0 = aC - alf x hc)

    // ------------------------------------------------------------------ rows
#pragma unroll 1
    for (int k = 0; k < NC; k++) {
        float4 t0, t1, t2;
        R.ld_tmp(k, t0, t1, t2);
        R.fence_tmp(t0, t1, t2);
        const bool on = (act >> k) & 1u;
        const V3 uJ = mk(t0.x, t2.z, t2.w);
        const float dist = t0.w + p0z;
        const V3 r = mk(t0.y - hc.x, t0.z - hc.y, t0.w - hc.z);
        // d2.y equals -d1.x up to round-off (A is symmetric): the record stores only d1.x and the solver reconstructs d2.y from
        // it, while the effective mass and right-hand side here use the d2.y pass 1 computed (a 1e-7 relative difference; writing
        // -d1.x here instead made the fma contractions of the row-storage instantiations differ, i.e. lost their bit-identity)
        const V3 d1 = mk(t1.x, t1.y, t1.z), d2 = mk(t1.w, t2.x, t2.y);
        // velocity of the contact point under the free rigid motion plus the new joint rates.  The rigid
        // field is (wf, velocity VC0 at C) with VC0 chosen so that the base origin gets v0 + dt a0:
        const V3 vp = VC + cross(wf, r) + uJ;
        // normal row
        const V3 rn = mk(r.y, -r.x, 0.f);
        const V3 Jn = mul(Ji, rn);
        const float Dn = invM + dot(rn, Jn);
        const float iDn = 1.f / Dn;
        const float pen = dist + P.slop;
        float verr = -vp.z, perr = 0.f;
        if (pen > 0.f) verr -= pen * inv_dt; else perr = -pen * P.erp2 * inv_dt;
        const float rhsn = (verr + perr) * iDn;
        // friction rows
        const V3 r1 = cross(r, d1), r2 = cross(r, d2);
        const V3 J1 = mul(Ji, r1), J2 = mul(Ji, r2);
        const float D1 = dot(d1, d1) * invM + dot(r1, J1), D2 = dot(d2, d2) * invM + dot(r2, J2);
        const float iD1 = 1.f / D1, iD2 = 1.f / D2;
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        R.st_rec(k, on ? make_float4(0.f, r.x, r.y, iDn) : z4, on ? make_float4(r.z, d1.x, d1.y, d1.z) : z4,
                 on ? make_float4(d2.x, d2.z, -dot(d1, vp) * iD1, -dot(d2, vp) * iD2) : z4, on ? make_float4(0.f, 0.f, iD1, iD2) : z4, on ? rhsn : 0.f);
    }
    R.fence_st();
    // hybrid rows: invD_n and rhs_n invD_n of every contact move from their parking words into registers (static indices: unrolled)
    float idn[Rows::REGN ? NC : 1], n1r[Rows::REGN ? NC : 1];
    if constexpr (Rows::REGN) {
#pragma unroll
        for (int k = 0; k < NC; k++) R.ld_regn(k, idn[k], n1r[k]);
#pragma unroll
        for (int k = 0; k < NC; k += 8) R.fence_regn8(idn + k, n1r + k);
#pragma unroll
        for (int k = 0; k < NC; k++) R.clr_lf(k);
        R.fence_st();
    }
    SNK_PHASE_MARK(1)

    // ------------------------------------------------------------------ projected Gauss-Seidel
    // The only serial dependence is the 6-vector (dw, dV); everything else of a row (loads, impulse
    // store, residual) is off that chain, and the loops are branch free so that the scheduler can
    // overlap it with the chain of the neighbouring rows.  The residual rule max (d D)^2 <= thr is
    // evaluated division free as  |d| <= sqrt(thr) invD  on every row.  A lane whose sweeps have ended
    // (converged, or masked from the start) is `frozen`: it keeps executing the warp's loop but commits
    // nothing, so its result is the one of the sweep at which the oracle's loop exits.
    V3 dw = mk(0.f, 0.f, 0.f), dV = mk(0.f, 0.f, 0.f);
    const float sthr = P.sthr, mu = P.mu; // kernel parameters: constant-bank operands, no register reads
    bool frozen = !commit;
    int sweeps = 0;
    // a frozen lane applies its (discarded) impulse changes through a ZERO inverse inertia: dw and dV stay bit-exact without any
    // per-row select or branch.  Nothing after the solver needs J^-1 or 1/M, so the lane's own copies are zeroed when it freezes.
    S3 Jg = Ji;
    float iM = invM;
#pragma unroll 1
    for (int it = 0; it < P.iters; it++) {
        if (ex_all(frozen)) break;
        float viol = 0.f; // max over the rows of |d| - sqrt(thr) invD (in the row's scaled units)
        if (frozen) { Jg.xx = 0.f; Jg.xy = 0.f; Jg.xz = 0.f; Jg.yy = 0.f; Jg.yz = 0.f; Jg.zz = 0.f; iM = 0.f; }
        {   // ---- normal rows; the record of row k+1 is fetched while row k is on the chain
            // one row: LN = normal impulse, RX / RY = lever arm, IDN = invD_n, N1 = rhs_n invD_n
#define SNK_NORMAL_ROW(K, LN, RX, RY, IDN, N1)                                            \
            {                                                                             \
                const float ln = (LN);                                                    \
                const float p = ln + (N1);                                                \
                float jd = fmaf(dw.x, (RY), dV.z);                                        \
                jd = fmaf(-dw.y, (RX), jd);                                               \
                const float sum = fmaxf(fmaf(-jd, (IDN), p), 0.f);                        \
                const float dd = sum - ln;                                                \
                R.st_ln((K), frozen ? ln : sum);                                          \
                const float t1 = (RY) * dd, t2 = -(RX) * dd; /* rn * dd */                \
                if (SNK_VAR_NDW == 0) {                                                   \
                    dw.x = fmaf(Jg.xx, t1, fmaf(Jg.xy, t2, dw.x));                        \
                    dw.y = fmaf(Jg.xy, t1, fmaf(Jg.yy, t2, dw.y));                        \
                    dw.z = fmaf(Jg.xz, t1, fmaf(Jg.yz, t2, dw.z));                        \
                } else {                                                                  \
                    dw.x = fmaf(Jg.xy, t2, fmaf(Jg.xx, t1, dw.x));                        \
                    dw.y = fmaf(Jg.yy, t2, fmaf(Jg.xy, t1, dw.y));                        \
                    dw.z = fmaf(Jg.yz, t2, fmaf(Jg.xz, t1, dw.z));                        \
                }                                                                         \
                dV.z = fmaf(dd, iM, dV.z);                                                \
                viol = fmaxf(viol, fmaf(-sthr, (IDN), fabsf(dd)));                        \
            }
            float4 nx; float nn = 0.f;
            R.ld_n(0, nx, nn);
            if constexpr (Rows::REGN) { // invD_n / rhs_n invD_n in registers: static contact index, fully unrolled
#pragma unroll
                for (int k = 0; k < NC; k++) {
                    R.fence4(nx);
                    const float4 x0 = nx;  // (ln, rx, ry, -)
                    if (k + 1 < NC) R.ld_n(k + 1, nx, nn);
                    SNK_NORMAL_ROW(k, x0.x, x0.y, x0.z, idn[k], n1r[k])
                }
            } else {
SNK_UNROLL(SNK_UNROLL_N)
                for (int k = 0; k < NC; k++) {
                    R.fence4(nx);
                    const float4 x0 = nx; const float n1 = nn;  // (ln, rx, ry, invD_n), rhs_n invD_n
                    R.ld_n((k + 1) & (NC - 1), nx, nn);
                    SNK_NORMAL_ROW(k, x0.x, x0.y, x0.z, x0.w, n1)
                }
                R.fence4(nx);
            }
#undef SNK_NORMAL_ROW
            R.fence_st();
        }
        {   // ---- friction pairs; row k+1 is fetched while row k is on the chain (the last two rows are peeled so that the
            // prefetch index never wraps: the addresses of a row's loads and stores are constant offsets from one running address)
            // x3 = (la, lb, invD_1, invD_2); d1 = (x1.y, x1.z, x1.w), d2 = (x2.x, -x1.y, x2.y)
            // The order of the operations in g1/g2 and in the dw update below is not arbitrary: different orders make ptxas
            // allocate registers differently, and every pair of source registers of one instruction that falls into the same
            // register bank costs an issue cycle.  tools/sass_bank_conflicts.py counts them in the SASS (profiles/README.md).
#define SNK_FRICTION_ROW(K)                                                                                                   \
            {                                                                                                                 \
                const float rx = x0.y, ry = x0.z, rz = x1.x;                                                                  \
                const float pa = x3.x + x2.z, pb = x3.y + x2.w, lim = mu * x0.x;                                              \
                /* u = dV + dw x r */                                                                                         \
                const float ux = SNK_VAR_U ? fmaf(dw.y, rz, fmaf(-dw.z, ry, dV.x)) : fmaf(-dw.z, ry, fmaf(dw.y, rz, dV.x));   \
                const float uy = SNK_VAR_U ? fmaf(dw.z, rx, fmaf(-dw.x, rz, dV.y)) : fmaf(-dw.x, rz, fmaf(dw.z, rx, dV.y));   \
                const float uz = SNK_VAR_U ? fmaf(dw.x, ry, fmaf(-dw.y, rx, dV.z)) : fmaf(-dw.y, rx, fmaf(dw.x, ry, dV.z));   \
                const float g1 = ex_dot3<SNK_VAR_G>(x1.y, ux, x1.z, uy, x1.w, uz);                                            \
                const float g2 = ex_dot3<SNK_VAR_G>(x2.x, ux, -x1.y, uy, x2.y, uz);                                           \
                float sa = fmaf(-g1, x3.z, pa), sb = fmaf(-g2, x3.w, pb);                                                     \
                if (CONE) { /* implicit cone: radial projection onto the disc of radius mu * lambda_n,                        \
                               s <- s min(1, lim / |s|)  (0/0 and lim/0 resolve to 1 through fminf) */                        \
                    const float sc = fminf(1.f, lim * ex_rsqrt_fast(fmaf(sa, sa, sb * sb)));                                  \
                    sa *= sc; sb *= sc;                                                                                       \
                } else {                                                                                                      \
                    sa = fminf(fmaxf(sa, -lim), lim);                                                                         \
                    sb = fminf(fmaxf(sb, -lim), lim);                                                                         \
                }                                                                                                             \
                const float da = sa - x3.x, db = sb - x3.y;                                                                   \
                R.st_lf((K), frozen ? x3.x : sa, frozen ? x3.y : sb);                                                         \
                const float fx = SNK_VAR_F ? fmaf(x1.y, da, x2.x * db) : fmaf(x2.x, db, x1.y * da);                           \
                const float fy = SNK_VAR_F ? fmaf(x1.z, da, -x1.y * db) : fmaf(-x1.y, db, x1.z * da);                         \
                const float fz = SNK_VAR_F ? fmaf(x1.w, da, x2.y * db) : fmaf(x2.y, db, x1.w * da);                           \
                /* r x f */                                                                                                   \
                const float tx = SNK_VAR_T ? fmaf(-rz, fy, ry * fz) : fmaf(ry, fz, -rz * fy);                                 \
                const float ty = SNK_VAR_T ? fmaf(-rx, fz, rz * fx) : fmaf(rz, fx, -rx * fz);                                 \
                const float tz = SNK_VAR_T ? fmaf(-ry, fx, rx * fy) : fmaf(rx, fy, -ry * fx);                                 \
                dV.x = fmaf(fx, iM, dV.x); dV.y = fmaf(fy, iM, dV.y); dV.z = fmaf(fz, iM, dV.z);                              \
                dw.x = ex_sum3<SNK_VAR_DW>(Jg.xx, tx, Jg.xy, ty, Jg.xz, tz, dw.x);                                            \
                dw.y = ex_sum3<SNK_VAR_DW>(Jg.xy, tx, Jg.yy, ty, Jg.yz, tz, dw.y);                                            \
                dw.z = ex_sum3<SNK_VAR_DW>(Jg.xz, tx, Jg.yz, ty, Jg.zz, tz, dw.z);                                            \
                /* (da D1 + db D2)^2 <= thr  <=>  |da invD2 + db invD1| <= sqrt(thr) invD1 invD2 */                           \
                viol = fmaxf(viol, fmaf(-sthr * x3.z, x3.w, fabsf(fmaf(da, x3.w, db * x3.z))));                               \
            }
            float4 n0, n1, n2_, n3;
            R.ld16(0, n0, n1, n2_, n3);
SNK_UNROLL(SNK_UNROLL_F)
            for (int k = 0; k < NC - 2; k++) {
                R.fence16(n0, n1, n2_, n3);
                const float4 x0 = n0, x1 = n1, x2 = n2_, x3 = n3;
                R.ld16(k + 1, n0, n1, n2_, n3);
                SNK_FRICTION_ROW(k)
            }
            {
                R.fence16(n0, n1, n2_, n3);
                const float4 x0 = n0, x1 = n1, x2 = n2_, x3 = n3;
                R.ld16(NC - 1, n0, n1, n2_, n3);
                SNK_FRICTION_ROW(NC - 2)
            }
            {
                R.fence16(n0, n1, n2_, n3);
                const float4 x0 = n0, x1 = n1, x2 = n2_, x3 = n3;
                SNK_FRICTION_ROW(NC - 1)
            }
#undef SNK_FRICTION_ROW
            R.fence_st();
        }
        if (!frozen) { sweeps++; frozen = (viol <= 0.f); }
    }
    out->iterations = sweeps;
    out->contacts = ex_popc(act);
    SNK_PHASE_MARK(2)

    // ------------------------------------------------------------------ new base velocity
    // rigid field after the solve: angular wf + dw, velocity VC + dV at C; base origin = field at -hc
    const V3 wN_u = wf + dw;
    const V3 vN_u = (VC + dV) - cross(wN_u, hc);
    // true base accelerations (before clamping, like the oracle): angular, and classical at the origin
    const V3 al0 = (wN_u - w0) * inv_dt;
    const V3 a0 = (vN_u - v0) * inv_dt;
    // clamp in body-0 axes (maxCoordinateVelocity)
    const M3 R0 = quat_to_m3(e.quat);
    V3 wb = mulT(R0, wN_u), vb = mulT(R0, vN_u);
    wb = mk(ex_clamp(wb.x, P.maxvel), ex_clamp(wb.y, P.maxvel), ex_clamp(wb.z, P.maxvel));
    vb = mk(ex_clamp(vb.x, P.maxvel), ex_clamp(vb.y, P.maxvel), ex_clamp(vb.z, P.maxvel));
    const V3 wN = mul(R0, wb), vN = mul(R0, vb);

    // ------------------------------------------------------------------ pass 2: base-ward, torques
    // Newton-Euler is linear in the accelerations, and the true ones differ from the reference ones of pass 1 by the base's
    // (a0, al0): the wrench of body i is the reference wrench plus  m (a0 + al0 x cc)  and  Iw al0.  Pass 2 therefore walks no
    // kinematics: it reads back what pass 1 kept of every body.  Only the torques (and, through them, the energy term of the
    // reward) depend on pass 2; they differ from a recomputed wrench at round-off.
#ifdef SNK_PASS2_RECOMPUTE
    // (build variant: the earlier pass 2, which walks the chain back and recomputes every wrench; the reference of
    // tests/test_gpu_setup_passes.py)
    {
        V3 SF = mk(0.f, 0.f, 0.f), SN = SF; // suffix wrench about the base origin
#pragma unroll 1
        for (int i = NB - 1; i >= 1; i--) {
            const int j = i - 1;
            const float q = slot(e, SNK_S_Q + j), qd = slot(e, SNK_S_QD + j), tg = R.tgt(j);
            float qds = P.kp * (tg - q) * inv_dt;
            qds = ex_clamp(qds, P.maxvel);
            const float qdd = (qds - qd) * inv_dt;
            // wrench of body i with the true accelerations
            V3 rc = mul(c.R, ld3(T.com[i]));
            V3 cc = c.p + rc;
            S3 Iw = world_inertia(T, i, c.R);
            V3 wxr = cross(c.w, rc);
            V3 vc = c.v + wxr;
            V3 ac = c.acc + cross(c.al, rc) + cross(c.w, wxr) + a0 + cross(al0, cc);
            V3 F, N;
            body_wrench(T, P, i, Iw, c.w, c.al + al0, vc, ac, &F, &N);
            SF = SF + F;
            SN = SN + cross(cc, F) + N;
#pragma unroll 1
            for (int k = T.cstart[i]; k < T.cstart[i + 1]; k++) { // a separated contact has a zero record: zero force
                float4 x0, x1, x2, x3;
                R.ld16(k, x0, x1, x2, x3);
                R.fence16(x0, x1, x2, x3);
                // contact force n ln + d1 la + d2 lb with d2 = (x2.x, -x1.y, x2.y); explicit fma so that every row-storage
                // instantiation rounds alike
                V3 f = mk(fmaf(x2.x, x3.y, x1.y * x3.x), fmaf(-x1.y, x3.y, x1.z * x3.x), fmaf(x2.y, x3.y, fmaf(x1.w, x3.x, x0.x))) * inv_dt;
                V3 r = mk(x0.y + hc.x, x0.z + hc.y, x1.x + hc.z); // back to the base origin
                SF = SF - f;
                SN = SN - cross(r, f);
            }
            V3 a = mul(c.R, ld3(T.jax[j]));
            const float tau = dot(a, SN - cross(c.p, SF)) + T.jdamp[j] * qd;
            if (commit) {
                slot(e, SNK_S_TAU + j) = tau;
                slot(e, SNK_S_QD + j) = qds;
                slot(e, SNK_S_Q + j) = q + qds * dt;
            }
            // step to the parent frame
            V3 wq = a * qd;
            c.w = c.w - wq;
            c.al = c.al - a * qdd - cross(c.w, wq);
            c.R = mulBT(c.R, joint_rot(T, j, q));
            V3 d = mul(c.R, ld3(T.jt[j]));
            V3 wxd = cross(c.w, d);
            c.p = c.p - d;
            c.v = c.v - wxd;
            c.acc = c.acc - cross(c.al, d) - cross(c.w, wxd);
        }
    }
#else
    {
        V3 SF = mk(0.f, 0.f, 0.f), SN = SF; // suffix wrench about the base origin
#pragma unroll 1
        for (int j = NJ - 1; j >= 0; j--) {
            const int i = j + 1;
            const float4 k0 = keep[j][0], k1 = keep[j][1], k2 = keep[j][2], k3 = keep[j][3], k4 = keep[j][4], k5 = keep[j][5];
            const float q = slot(e, SNK_S_Q + j), qd = slot(e, SNK_S_QD + j), tg = R.tgt(j);
            float qds = P.kp * (tg - q) * inv_dt;
            qds = ex_clamp(qds, P.maxvel);
            // wrench of body i with the true accelerations
            S3 Iw; Iw.xx = k0.x; Iw.xy = k0.y; Iw.xz = k0.z; Iw.yy = k0.w; Iw.yz = k1.x; Iw.zz = k1.y;
            const V3 a = mk(k1.z, k1.w, k2.x), p = mk(k2.y, k2.z, k2.w), cc = mk(k3.x, k3.y, k3.z);
            const V3 F = mk(k3.w, k4.x, k4.y) + (a0 + cross(al0, cc)) * T.mass[i];
            const V3 N = mk(k4.z, k4.w, k5.x) + mul(Iw, al0);
            SF = SF + F;
            SN = SN + cross(cc, F) + N;
#pragma unroll 1
            for (int k = T.cstart[i]; k < T.cstart[i + 1]; k++) { // a separated contact has a zero record: zero force
                float4 x0, x1, x2, x3;
                R.ld16(k, x0, x1, x2, x3);
                R.fence16(x0, x1, x2, x3);
                // contact force n ln + d1 la + d2 lb with d2 = (x2.x, -x1.y, x2.y); explicit fma so that every row-storage
                // instantiation rounds alike
                V3 f = mk(fmaf(x2.x, x3.y, x1.y * x3.x), fmaf(-x1.y, x3.y, x1.z * x3.x), fmaf(x2.y, x3.y, fmaf(x1.w, x3.x, x0.x))) * inv_dt;
                V3 r = mk(x0.y + hc.x, x0.z + hc.y, x1.x + hc.z); // back to the base origin
                SF = SF - f;
                SN = SN - cross(r, f);
            }
            const float tau = dot(a, SN - cross(p, SF)) + T.jdamp[j] * qd;
            if (commit) {
                slot(e, SNK_S_TAU + j) = tau;
                slot(e, SNK_S_QD + j) = qds;
                slot(e, SNK_S_Q + j) = q + qds * dt;
            }
        }
    }
#endif

    // ------------------------------------------------------------------ finish: Fz, base integration
    {   // reaction force of joint 0 (kdl_dummy_root -> base), z of link `base` (snake.py:202-206)
        const float nv = sqrtf(dot(v0, v0));
        const float rm = T.rootm, kl = P.kl + P.kl * nv;
        V3 f = mk(rm * P.g[0] - rm * v0.x * kl - rm * (vN.x - v0.x) * inv_dt, rm * P.g[1] - rm * v0.y * kl - rm * (vN.y - v0.y) * inv_dt,
                  rm * P.g[2] - rm * v0.z * kl - rm * (vN.z - v0.z) * inv_dt);
        if (commit) slot(e, SNK_S_FZ) = dot(mul(R0, ld3(T.fzax)), f);
    }
    if (commit) {
    e.vel[0] = vN.x; e.vel[1] = vN.y; e.vel[2] = vN.z;
    e.omg[0] = wN.x; e.omg[1] = wN.y; e.omg[2] = wN.z;
    e.pos[0] += vN.x * dt; e.pos[1] += vN.y * dt; e.pos[2] += vN.z * dt;
    {   // quaternion exponential map, q <- exp(w dt / 2) * q, normalised
        const float ang = sqrtf(dot(wN, wN));
        float sc, sn, cw;
        ex_sincos(0.5f * ang * dt, &sn, &cw);
        if (ang < 0.001f) sc = 0.5f * dt - dt * dt * dt * 0.020833333333f * ang * ang;
        else sc = sn / ang;
        const float ax = wN.x * sc, ay = wN.y * sc, az = wN.z * sc;
        const float* q = e.quat;
        float x = cw * q[0] + ax * q[3] + ay * q[2] - az * q[1];
        float y = cw * q[1] + ay * q[3] + az * q[0] - ax * q[2];
        float z = cw * q[2] + az * q[3] + ax * q[1] - ay * q[0];
        float w = cw * q[3] - ax * q[0] - ay * q[1] - az * q[2];
        const float in = ex_rsqrt(x * x + y * y + z * z + w * w);
        e.quat[0] = x * in; e.quat[1] = y * in; e.quat[2] = z * in; e.quat[3] = w * in;
    }
    }
    SNK_PHASE_MARK(3)
}

// mean z of the checkSnakeHeight points (snake.py:237-245) of the current state: a z-only walk
// (third row of every frame), used where no tick follows.
SNK_HD float ex_height(const ExTables& T, const ExEnv& e) {
    const M3 R0 = quat_to_m3(e.quat);
    V3 r3 = mk(R0.m[6], R0.m[7], R0.m[8]); // third row of the current frame
    float z = e.pos[2];
    float hsum = z + r3.x * T.hpt[0][0] + r3.y * T.hpt[0][1] + r3.z * T.hpt[0][2];
#pragma unroll 1
    for (int i = 1; i < NB; i++) {
        const int j = i - 1;
        z += r3.x * T.jt[j][0] + r3.y * T.jt[j][1] + r3.z * T.jt[j][2];
        const M3 Mj = joint_rot(T, j, slot(e, SNK_S_Q + j));
        r3 = mulT(Mj, r3);
        hsum += z + r3.x * T.hpt[i][0] + r3.y * T.hpt[i][1] + r3.z * T.hpt[i][2];
    }
    return hsum * (1.f / NB);
}

// world COM positions of URDF links arange(0,49,3) of the current state as [x0..x16 | y0..y16 | z0..z16]
// (Snake.getLinkPositions, snake.py:138-146; the points checkSnakeHeight averages): mode='test' info stream only
SNK_HD void ex_link_positions(const ExTables& T, const ExEnv& e, float* out) {
    M3 R = quat_to_m3(e.quat);
    V3 p = ld3(e.pos);
#pragma unroll 1
    for (int i = 0; i < NB; i++) {
        if (i > 0) {
            const int j = i - 1;
            p = p + mul(R, ld3(T.jt[j]));
            R = mul(R, joint_rot(T, j, slot(e, SNK_S_Q + j)));
        }
        const V3 w = p + mul(R, ld3(T.hpt[i]));
        out[i] = w.x; out[NB + i] = w.y; out[2 * NB + i] = w.z;
    }
}

// -----------------------------------------------------------------------------------------------
// task logic around the tick: one SubprocVecEnv.step of one environment (oracle: env_step).
// S.tgt[.][tid] must hold the 16 joint targets (checkBound + createAction + scaling already applied).
// On return the state slots and e.pos.. hold the post-step (post-reset when done) state.
// -----------------------------------------------------------------------------------------------
struct ExStepOut { float rew; int done, ticks, iters, bad; };

SNK_HD float ex_obs_of(const ExEnv& e, int k) { // snake.py:209-217
    if (k < 16) return slot(e, SNK_S_Q + k);
    if (k < 32) return slot(e, SNK_S_QD + k - 16);
    if (k < 48) return slot(e, SNK_S_TAU + k - 32);
    if (k < 51) return e.pos[k - 48];
    if (k < 55) return e.quat[k - 51];
    return slot(e, SNK_S_FZ);
}
SNK_HD bool ex_finite(float x) { return fabsf(x) <= 3.402823466e38f; } // false for inf and nan

SNK_HD void ex_load_base(ExEnv& e) {
#pragma unroll
    for (int k = 0; k < 3; k++) { e.pos[k] = slot(e, SNK_S_POS + k); e.vel[k] = slot(e, SNK_S_VEL + k); e.omg[k] = slot(e, SNK_S_OMEGA + k); }
#pragma unroll
    for (int k = 0; k < 4; k++) e.quat[k] = slot(e, SNK_S_QUAT + k);
}
SNK_HD void ex_store_base(const ExEnv& e) {
#pragma unroll
    for (int k = 0; k < 3; k++) { slot(e, SNK_S_POS + k) = e.pos[k]; slot(e, SNK_S_VEL + k) = e.vel[k]; slot(e, SNK_S_OMEGA + k) = e.omg[k]; }
#pragma unroll
    for (int k = 0; k < 4; k++) slot(e, SNK_S_QUAT + k) = e.quat[k];
}

// progress of one environment through its env-step (snake.py:274-306): kept in registers between ticks
struct ExRun { float xprev, e2, height; int counter, iters; bool end_height, have_height; };

template <class Rows>
SNK_HD void ex_step_begin(const KParams& P, const Rows& R, const ExEnv& e, ExRun* r) {
    r->xprev = e.pos[0]; // self._observation[48], vec-wrapper semantics (Q8)
    float e2 = 0.f;
#pragma unroll 1
    for (int j = 0; j < NJ; j++) { const float d = R.tgt(j) - slot(e, SNK_S_Q + j); e2 += d * d; }
    r->e2 = e2; r->height = 0.f; r->counter = 0; r->iters = 0; r->end_height = false; r->have_height = false;
}

// At most one physics tick.  Warp convergent: every lane of the warp calls it; `have` says whether the lane
// owns an environment.  Returns true (only for lanes with `have`) when the tick loop of snake.py:284-304 has
// ended for the lane's environment.
template <bool CONE, class Rows>
SNK_HD bool ex_step_advance(const ExTables& T, const KParams& P, const Rows& R, ExEnv& e, bool have, ExRun* r) {
    const bool need = have && (sqrtf(r->e2) > P.errthr); // checkFeedback (snake.py:228-235); false: zero-tick step (Q5)
    bool aborted;
    ExTickOut to;
    ex_tick<CONE>(T, P, R, e, need, r->counter > 0, &aborted, &to);
    if (!have) return false;
    if (!need) return true;
    if (aborted) { r->end_height = true; r->height = to.height; r->have_height = true; return true; } // the previous tick lifted the snake
    r->iters += to.iterations;
    r->counter++;
    r->e2 = to.err2_next;
    return r->counter >= P.maxticks || !(sqrtf(r->e2) > P.errthr); // `counter > 40`
}

SNK_HD void ex_step_end(const ExTables& T, const KParams& P, ExEnv& e, const ExRun& run, ExStepOut* o) {
    const float xprev = run.xprev;
    const int counter = run.counter, iters = run.iters;
    const bool end_height = run.end_height;
    const float height = run.have_height ? run.height : ex_height(T, e);
    // non-finite guard, energy (snake.py:336-341)
    bool bad = false;
    float energy = 0.f;
#pragma unroll
    for (int k = 0; k < 3; k++) bad |= !ex_finite(e.pos[k]) || !ex_finite(e.vel[k]) || !ex_finite(e.omg[k]);
#pragma unroll
    for (int k = 0; k < 4; k++) bad |= !ex_finite(e.quat[k]);
#pragma unroll 1
    for (int j = 0; j < NJ; j++) {
        const float q = slot(e, SNK_S_Q + j), qd = slot(e, SNK_S_QD + j), tau = slot(e, SNK_S_TAU + j);
        bad |= !ex_finite(q) || !ex_finite(qd) || !ex_finite(tau);
        energy += qd * tau * P.edt;
    }
    const float fz = slot(e, SNK_S_FZ);
    float ret = slot(e, SNK_S_RET), len = slot(e, SNK_S_LEN);
    bad |= !ex_finite(fz) || !ex_finite(ret) || !ex_finite(len);
    // calculateReward (SnakeGymEnv.py:90-97), checkTermination (SnakeGymEnv.py:99-103)
    float r = P.alpha * (e.pos[0] - xprev) + ((fabsf(fz) > P.colf) ? P.colpen : 0.f) - P.beta * fabsf(e.pos[1] - 0.f) - P.gamma * energy;
    bool d = (fabsf(ex_obs_of(e, P.tjoint)) > P.tang) || (height > P.hthr) || end_height;
    if (bad) {
        d = true; r = P.donepen;
#pragma unroll 1
        for (int k = 0; k < SNK_STATE_STRIDE; k++) slot(e, k) = 0.f;
        ret = 0.f; len = 0.f;
    } else if (d) r += P.donepen;
    ret += r; len += 1.f;
    if (d) { // in-step reset + worker reset: the returned obs is the post-reset one (multiprocessing_env.py:14-15)
#pragma unroll
        for (int k = 0; k < 3; k++) { e.pos[k] = 0.f; e.vel[k] = 0.f; e.omg[k] = 0.f; e.quat[k] = 0.f; }
        e.quat[3] = 1.f;
#pragma unroll 1
        for (int j = 0; j < NJ; j++) { slot(e, SNK_S_Q + j) = 0.f; slot(e, SNK_S_QD + j) = 0.f; if (!P.stale) slot(e, SNK_S_TAU + j) = 0.f; }
        if (!P.stale) slot(e, SNK_S_FZ) = 0.f;
        ret = 0.f; len = 0.f;
    }
    slot(e, SNK_S_RET) = ret; slot(e, SNK_S_LEN) = len;
    ex_store_base(e);
    o->rew = r; o->done = d ? 1 : 0; o->ticks = counter; o->iters = iters; o->bad = bad ? 1 : 0;
}

template <bool CONE, class Rows>
SNK_HD void ex_env_step(const ExTables& T, const KParams& P, const Rows& R, ExEnv& e, ExStepOut* o) {
    ExRun run;
    ex_step_begin(P, R, e, &run);
    while (!ex_step_advance<CONE>(T, P, R, e, true, &run)) {}
    ex_step_end(T, P, e, run, o);
}
