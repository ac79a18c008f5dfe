// Two-lines-per-thread Stockham passes on packed fp32 pairs (FADD2 / FMUL2 / FFMA2 of sm_100a).
//
// The fused SENSE passes of fft_il.cuh issue ~70 instructions per grid point, half of them scalar
// fp32 arithmetic, and run at IPC 2.2-2.3 of 4: issue bound at 43 % of the DRAM peak
// (profiles/r01_s6_state_cfg3.md).  Blackwell executes add/mul/fma on two fp32 lanes of a 64-bit
// register pair with ONE issue slot (tools/micro/ffma2_bench.cu: same 128 lane-ops/clk/SM, half the
// instructions; ptxas folds broadcast scalars, immediates and negated addends into the operand
// modifiers).  Here a thread owns the SAME butterfly of two neighbouring lines of the 16-line tile:
// the pair (line 2p, line 2p+1) is 16 contiguous bytes in global memory, its real parts form one
// packed register and its imaginary parts another, so every scalar operation of the radix
// butterflies becomes one packed operation and the twiddles (which depend on the position only)
// are shared.  Shared memory holds split planes re[pos][16] / im[pos][16]: a pair is one 8-byte
// word, four consecutive positions of one warp are 256 contiguous bytes (conflict free, no padding).
//
// Same Stockham recurrence and stage sequencing as fft_core.cuh (the emulation harness runs these
// bodies on the CPU against numpy, tests/test_fft_emulation.py).
#pragma once
#include "fft_il.cuh"
#include "pk2.cuh"

namespace ib200 {

// complex values of two lines: x = (re0, re1), y = (im0, im1)
struct cpk { pk2 x, y; };
IB_HD cpk k_mk(pk2 x, pk2 y) { cpk r; r.x = x; r.y = y; return r; }
IB_HD cpk k_zero() { return k_mk(p_make(0.f, 0.f), p_make(0.f, 0.f)); }
IB_HD cpk k_add(cpk a, cpk b) { return k_mk(p_add(a.x, b.x), p_add(a.y, b.y)); }
IB_HD cpk k_sub(cpk a, cpk b) { return k_mk(p_sub(a.x, b.x), p_sub(a.y, b.y)); }
IB_HD cpk k_swap(cpk a) { return k_mk(a.y, a.x); }
// a + (-i)*d  and  a - (-i)*d      ((-i)*(dx + i dy) = dy - i dx)
IB_HD cpk k_add_mi(cpk a, cpk d) { return k_mk(p_add(a.x, d.y), p_sub(a.y, d.x)); }
IB_HD cpk k_sub_mi(cpk a, cpk d) { return k_mk(p_sub(a.x, d.y), p_add(a.y, d.x)); }
// u * w for a scalar complex w shared by both lines: 4 packed operations
IB_HD cpk k_mul_w(cpk u, c64 w) {
    const pk2 wr = p_bc(w.x), wi = p_bc(w.y);
    return k_mk(p_sub(p_mul(u.x, wr), p_mul(u.y, wi)), p_fma(u.x, wi, p_mul(u.y, wr)));
}
// u * (c - i s) for compile-time c, s
IB_HD cpk k_mul_cs(cpk u, float c, float s) {
    return k_mk(p_fmac(s, u.y, p_scale(c, u.x)), p_fmac(-s, u.x, p_scale(c, u.y)));
}

// ---- forward DFTs of a register-resident vector of line pairs (no negations: adds, subs, fmas) ---
template <int R> struct DftK {
    // odd prime R, same pairing as Dft<R> of fft_core.cuh
    IB_HD static void run(cpk (&u)[R]) {
        constexpr int H = (R - 1) / 2;
        cpk a[H], b[H];
#pragma unroll
        for (int j = 0; j < H; ++j) { a[j] = k_add(u[j + 1], u[R - 1 - j]); b[j] = k_sub(u[j + 1], u[R - 1 - j]); }
        const cpk x0 = u[0];
        cpk s0 = x0;
#pragma unroll
        for (int j = 0; j < H; ++j) s0 = k_add(s0, a[j]);
        u[0] = s0;
#pragma unroll
        for (int k = 1; k <= H; ++k) {
            cpk ck = x0, sk;
#pragma unroll
            for (int j = 1; j <= H; ++j) {
                const int m = (j * k) % R;
                const float cv = m <= H ? Trig<R>::c(m - 1) : Trig<R>::c(R - m - 1);
                const float sv = m <= H ? Trig<R>::s(m - 1) : -Trig<R>::s(R - m - 1);
                ck.x = p_fmac(cv, a[j - 1].x, ck.x); ck.y = p_fmac(cv, a[j - 1].y, ck.y);
                if (j == 1) { sk.x = p_scale(sv, b[0].x); sk.y = p_scale(sv, b[0].y); }
                else { sk.x = p_fmac(sv, b[j - 1].x, sk.x); sk.y = p_fmac(sv, b[j - 1].y, sk.y); }
            }
            u[k] = k_add_mi(ck, sk);                        // ck - i*sk
            u[R - k] = k_sub_mi(ck, sk);                    // ck + i*sk
        }
    }
};

template <> struct DftK<2> {
    IB_HD static void run(cpk (&u)[2]) { const cpk a = u[0], b = u[1]; u[0] = k_add(a, b); u[1] = k_sub(a, b); }
};

template <> struct DftK<4> {
    IB_HD static void run(cpk (&u)[4]) {
        const cpk t0 = k_add(u[0], u[2]), t1 = k_sub(u[0], u[2]);
        const cpk t2 = k_add(u[1], u[3]), d = k_sub(u[1], u[3]);
        u[0] = k_add(t0, t2); u[2] = k_sub(t0, t2);
        u[1] = k_add_mi(t1, d); u[3] = k_sub_mi(t1, d);
    }
};

template <> struct DftK<8> {
    IB_HD static void run(cpk (&u)[8]) {
        cpk e[4] = {u[0], u[2], u[4], u[6]}, o[4] = {u[1], u[3], u[5], u[7]};
        DftK<4>::run(e); DftK<4>::run(o);
        const float h = 0.70710678118654752f;
        u[0] = k_add(e[0], o[0]); u[4] = k_sub(e[0], o[0]);
        // o1 * (1 - i)/sqrt2 = h*(ox + oy) + i*h*(oy - ox)
        { const pk2 s = p_add(o[1].x, o[1].y), d = p_sub(o[1].y, o[1].x);
          u[1] = k_mk(p_fmac(h, s, e[1].x), p_fmac(h, d, e[1].y)); u[5] = k_mk(p_fmac(-h, s, e[1].x), p_fmac(-h, d, e[1].y)); }
        u[2] = k_add_mi(e[2], o[2]); u[6] = k_sub_mi(e[2], o[2]);
        // o3 * (-1 - i)/sqrt2 = h*(oy - ox) - i*h*(ox + oy)
        { const pk2 s = p_add(o[3].x, o[3].y), d = p_sub(o[3].y, o[3].x);
          u[3] = k_mk(p_fmac(h, d, e[3].x), p_fmac(-h, s, e[3].y)); u[7] = k_mk(p_fmac(-h, d, e[3].x), p_fmac(h, s, e[3].y)); }
    }
};

template <> struct DftK<16> {
    IB_HD static void run(cpk (&u)[16]) {
        cpk y[4][4];
#pragma unroll
        for (int n2 = 0; n2 < 4; ++n2) {
            cpk t[4] = {u[n2], u[4 + n2], u[8 + n2], u[12 + n2]};
            DftK<4>::run(t);
#pragma unroll
            for (int k1 = 0; k1 < 4; ++k1) y[n2][k1] = t[k1];
        }
        const float c1 = 0.92387953251128674f, s1 = 0.38268343236508977f, h = 0.70710678118654752f;
        // w16^m = cos(2 pi m/16) - i sin(2 pi m/16)
        y[1][1] = k_mul_cs(y[1][1], c1, s1);
        y[1][2] = k_mul_cs(y[1][2], h, h);
        y[1][3] = k_mul_cs(y[1][3], s1, c1);
        y[2][1] = k_mul_cs(y[2][1], h, h);
        y[2][2] = k_mk(y[2][2].y, p_sub(p_make(0.f, 0.f), y[2][2].x));   // * -i
        y[2][3] = k_mul_cs(y[2][3], -h, h);
        y[3][1] = k_mul_cs(y[3][1], s1, c1);
        y[3][2] = k_mul_cs(y[3][2], -h, h);
        y[3][3] = k_mul_cs(y[3][3], -c1, -s1);             // w16^9
#pragma unroll
        for (int k1 = 0; k1 < 4; ++k1) {
            cpk t[4] = {y[0][k1], y[1][k1], y[2][k1], y[3][k1]};
            DftK<4>::run(t);
#pragma unroll
            for (int k2 = 0; k2 < 4; ++k2) u[k1 + 4 * k2] = t[k2];
        }
    }
};

// ---- shared-memory tile: split planes, 16 floats per position -------------------------------------
static const int kPkPairs = kSpecL / 2;                              // line pairs per tile
IB_HD size_t pk_buf_floats(int n) { return (size_t)2 * n * kSpecL; }  // one buffer (re plane + im plane)

template <int N>
IB_HD cpk pk_lds(const float *buf, int pos, int lp) {
    const pk2 *re = reinterpret_cast<const pk2 *>(buf + pos * kSpecL) + lp;
    const pk2 *im = reinterpret_cast<const pk2 *>(buf + N * kSpecL + pos * kSpecL) + lp;
    return k_mk(*re, *im);
}
template <int N>
IB_HD void pk_sts(float *buf, int pos, int lp, cpk v) {
    reinterpret_cast<pk2 *>(buf + pos * kSpecL)[lp] = v.x;
    reinterpret_cast<pk2 *>(buf + N * kSpecL + pos * kSpecL)[lp] = v.y;
}

// two neighbouring complex words of global memory <-> one line pair
IB_HD cpk pk_from_f4(float r0, float i0, float r1, float i1) { return k_mk(p_make(r0, r1), p_make(i0, i1)); }

struct PkQuad { float r0, i0, r1, i1; };
IB_HD PkQuad pk_gld(const c64 *p) {
#ifdef __CUDA_ARCH__
    const float4 v = *reinterpret_cast<const float4 *>(p);
    PkQuad q; q.r0 = v.x; q.i0 = v.y; q.r1 = v.z; q.i1 = v.w; return q;
#else
    PkQuad q; q.r0 = p[0].x; q.i0 = p[0].y; q.r1 = p[1].x; q.i1 = p[1].y; return q;
#endif
}
IB_HD void pk_gst(c64 *p, cpk v) {
#ifdef __CUDA_ARCH__
    *reinterpret_cast<float4 *>(p) = make_float4(p_lo(v.x), p_lo(v.y), p_hi(v.x), p_hi(v.y));
#else
    p[0] = h_mk(p_lo(v.x), p_lo(v.y)); p[1] = h_mk(p_hi(v.x), p_hi(v.y));
#endif
}

// ---- one Stockham stage over line pairs ---------------------------------------------------------
// CTX supplies: int npairs; const c64 *tw; cpk gload(int lp, int pos); void gstore(int lp, int pos, cpk).
// Twiddles w^(s*k*STEP) are read from the table directly (s*k*STEP < N): R-1 independent cached
// loads instead of one load and a dependent chain of complex multiplications.
template <int N, int R, int P, bool SRC_G, bool DST_G, class CTX>
IB_HD void pk_stage_item(const CTX &c, const float *sin_, float *sout, int idx) {
    constexpr int T = N / R, STEP = N / (P * R);
    const int lp = idx & (kPkPairs - 1), b = idx >> 3;
    if (lp >= c.npairs) return;
    const int k = P == 1 ? 0 : b % P;
    cpk u[R];
#pragma unroll
    for (int s = 0; s < R; ++s) {
        const int pos = b + s * T;
        u[s] = SRC_G ? c.gload(lp, pos) : pk_lds<N>(sin_, pos, lp);
    }
    if (P > 1) {
        c64 pw[R];
#pragma unroll
        for (int s = 1; s < R; ++s) pw[s] = c.tw[s * k * STEP];
#pragma unroll
        for (int s = 1; s < R; ++s) u[s] = k_mul_w(u[s], pw[s]);
    }
    DftK<R>::run(u);
    const int o0 = (b - k) * R + k;
#pragma unroll
    for (int q = 0; q < R; ++q) {
        const int pos = o0 + q * P;
        if (DST_G) c.gstore(lp, pos, u[q]);
        else pk_sts<N>(sout, pos, lp, u[q]);
    }
}

// NT > 0: the CTA has exactly NT threads; the rounds of a stage are unrolled so that the loads of
// neighbouring rounds overlap.  NT == 0: runtime thread count (emulation).
template <int N, int R, int P, bool SRC_G, bool DST_G, int NT, class CTX>
IB_HD void pk_stage(const CTX &c, const float *sin_, float *sout, int tid, int nt) {
    constexpr int T = N / R, ITEMS = kPkPairs * T;
    if (NT > 0) {
        constexpr int K = NT > 0 ? (ITEMS + NT - 1) / NT : 1;
#pragma unroll
        for (int r = 0; r < K; ++r) {
            const int idx = tid + r * NT;
            if (idx < ITEMS) pk_stage_item<N, R, P, SRC_G, DST_G>(c, sin_, sout, idx);
        }
    } else {
        for (int idx = tid; idx < ITEMS; idx += nt) pk_stage_item<N, R, P, SRC_G, DST_G>(c, sin_, sout, idx);
    }
}

// stages 1..3 of one tile; SRC/DST of the ends are the context's global accessors unless
// LAST_TO_SMEM (the combine pass post-processes the result in shared memory).  Returns the buffer
// holding the result when LAST_TO_SMEM.
template <int N, int R0, int R1, int R2, bool LAST_TO_SMEM, int NT, class CTX>
IB_HD float *pk_run_stages(const CTX &c, float *bufA, int tid, int nt) {
    constexpr bool THREE = R2 > 1;
    float *bufB = bufA + pk_buf_floats(N);
    pk_stage<N, R0, 1, true, false, NT>(c, nullptr, bufA, tid, nt);
    IB_SYNC();
    if (THREE) {
        pk_stage<N, R1, R0, false, false, NT>(c, bufA, bufB, tid, nt);
        IB_SYNC();
        if (LAST_TO_SMEM) { pk_stage<N, THREE ? R2 : R1, R0 * R1, false, false, NT>(c, bufB, bufA, tid, nt); IB_SYNC(); return bufA; }
        pk_stage<N, THREE ? R2 : R1, R0 * R1, false, true, NT>(c, bufB, nullptr, tid, nt);
        return nullptr;
    }
    if (LAST_TO_SMEM) { pk_stage<N, R1, R0, false, false, NT>(c, bufA, bufB, tid, nt); IB_SYNC(); return bufB; }
    pk_stage<N, R1, R0, false, true, NT>(c, bufA, nullptr, tid, nt);
    return nullptr;
}
IB_HD size_t pk_smem_floats(int n, bool three, bool last_to_smem) {
    return pk_buf_floats(n) * ((three || last_to_smem) ? 2 : 1);
}

// ---- strided passes (y and z) on the interleaved grid ---------------------------------------------
template <bool SWAP_IN, bool SWAP_OUT>
struct PkIlCtx {
    const c64 *gin; c64 *gout; const c64 *tw;
    unsigned pstride;
    int in0; unsigned inlen; int out0; unsigned outlen;
    static constexpr int npairs = kPkPairs;
    IB_HD cpk gload(int lp, int pos) const {
        if ((unsigned)(pos - in0) >= inlen) return k_zero();
        const PkQuad q = pk_gld(gin + (uint64_t)(unsigned)pos * pstride + (unsigned)(2 * lp));
        return SWAP_IN ? pk_from_f4(q.i0, q.r0, q.i1, q.r1) : pk_from_f4(q.r0, q.i0, q.r1, q.i1);
    }
    IB_HD void gstore(int lp, int pos, cpk v) const {
        if ((unsigned)(pos - out0) >= outlen) return;
        pk_gst(gout + (uint64_t)(unsigned)pos * pstride + (unsigned)(2 * lp), SWAP_OUT ? k_swap(v) : v);
    }
};

template <int N, int R0, int R1, int R2, bool SWAP_IN, bool SWAP_OUT, int NT>
IB_HD void fft_pk_pass_body(const IlPassArgs &a, float *bufA, int64_t block, int tid, int nt) {
    const int64_t tiles = a.inner / kSpecL;
    const int64_t o = block / tiles, s0 = (block % tiles) * kSpecL;
    PkIlCtx<SWAP_IN, SWAP_OUT> c;
    c.gin = a.x + o * a.outer_stride + s0; c.gout = a.x + o * a.outer_stride + s0;
    c.tw = a.tw; c.pstride = a.pstride;
    c.in0 = a.in0; c.inlen = (unsigned)(a.in1 - a.in0); c.out0 = a.out0; c.outlen = (unsigned)(a.out1 - a.out0);
    pk_run_stages<N, R0, R1, R2, false, NT>(c, bufA, tid, nt);
}

// ---- persistent, prefetching form of the strided passes ---------------------------------------------
// The one-shot kernel above keeps 2 CTAs of 8 warps per SM whose load, butterfly and store phases
// seldom overlap: ~26 KB in flight per SM on average where HBM needs ~35 KB (Little), 42-46 % of the
// DRAM peak although a pure copy with the same 128-byte/22 MB access pattern reaches 85-95 %
// (tools/micro/strided_copy.cu).  Here a CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ...; the
// raw input of the NEXT tile streams into a second shared buffer with cp.async (only the positions of
// the input window) while the current tile runs its second and third stage, so loads are in flight all
// the time.  Shared memory stays at two buffers per CTA because the middle stage works in place
// (every thread reads its butterflies into registers, barrier, writes them back).
struct PkPrefCtxBase {
    const c64 *raw;                    // prefetched tile: raw[pos*16 + line], complex words as in global memory
    c64 *gout; const c64 *tw;
    unsigned pstride;
    int in0; unsigned inlen; int out0; unsigned outlen;
    static constexpr int npairs = kPkPairs;
};
template <bool SWAP_IN, bool SWAP_OUT>
struct PkPrefCtx : PkPrefCtxBase {
    IB_HD cpk gload(int lp, int pos) const {
        if ((unsigned)(pos - in0) >= inlen) return k_zero();
        const PkQuad q = pk_gld(raw + pos * kSpecL + 2 * lp);
        return SWAP_IN ? pk_from_f4(q.i0, q.r0, q.i1, q.r1) : pk_from_f4(q.r0, q.i0, q.r1, q.i1);
    }
    IB_HD void gstore(int lp, int pos, cpk v) const {
        if ((unsigned)(pos - out0) >= outlen) return;
        pk_gst(gout + (uint64_t)(unsigned)pos * pstride + (unsigned)(2 * lp), SWAP_OUT ? k_swap(v) : v);
    }
};

IB_HD const c64 *pkp_tile_base(const IlPassArgs &a, int64_t tile) {
    const int64_t tiles = a.inner / kSpecL;
    return a.x + (tile / tiles) * a.outer_stride + (tile % tiles) * kSpecL;
}

// stream the input window of `tile` into raw[] (16-byte chunks, 8 per position)
// window of a tile along the transformed axis: input window when `input`, else output window
IB_HD void pkp_tile_window(const IlPassArgs &a, int64_t tile, bool input, int &lo, int &hi) {
    lo = input ? a.in0 : a.out0; hi = input ? a.in1 : a.out1;
    if (a.win && a.win_mode == (input ? 2 : 1)) {
        const int64_t tiles = a.inner / kSpecL;
        const int64_t p = ((tile % tiles) * kSpecL) / a.win_div;
        const int wl = a.win[2 * p], wh = a.win[2 * p + 1];
        lo = wl > lo ? wl : lo; hi = wh < hi ? wh : hi;
        if (hi < lo) hi = lo;
    }
}

IB_HD void pkp_prefetch(const IlPassArgs &a, int64_t tile, c64 *raw, int tid, int nt) {
    const c64 *g = pkp_tile_base(a, tile);
    int in0, in1;
    pkp_tile_window(a, tile, true, in0, in1);
    const int chunks = (in1 - in0) * kPkPairs;
    for (int i = tid; i < chunks; i += nt) {
        const int pos = in0 + (i >> 3), ch = i & 7;
        const c64 *src = g + (uint64_t)(unsigned)pos * a.pstride + 2 * ch;
        c64 *dst = raw + pos * kSpecL + 2 * ch;
#ifdef __CUDA_ARCH__
        const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(src) : "memory");
#else
        dst[0] = src[0]; dst[1] = src[1];
#endif
    }
#ifdef __CUDA_ARCH__
    asm volatile("cp.async.commit_group;\n" ::: "memory");
#endif
}
IB_HD void pkp_wait() {
#ifdef __CUDA_ARCH__
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
#endif
}

// middle stage in place: all butterflies of the tile are read into registers before any is written
template <int N, int R, int P, int NT, class CTX>
IB_HD void pk_stage_inplace(const CTX &c, float *buf, int tid, int nt) {
    constexpr int T = N / R, ITEMS = kPkPairs * T, STEP = N / (P * R);
#ifdef __CUDA_ARCH__
    constexpr int K = (ITEMS + NT - 1) / (NT > 0 ? NT : 1);
    cpk u[K][R];
#pragma unroll
    for (int s = 0; s < K; ++s) {
        const int idx = tid + s * NT;
        if (idx < ITEMS) {
            const int lp = idx & (kPkPairs - 1), b = idx >> 3;
            const int k = b % P;
#pragma unroll
            for (int r = 0; r < R; ++r) u[s][r] = pk_lds<N>(buf, b + r * T, lp);
            c64 pw[R];
#pragma unroll
            for (int r = 1; r < R; ++r) pw[r] = c.tw[r * k * STEP];
#pragma unroll
            for (int r = 1; r < R; ++r) u[s][r] = k_mul_w(u[s][r], pw[r]);
            DftK<R>::run(u[s]);
        }
    }
    __syncthreads();
#pragma unroll
    for (int s = 0; s < K; ++s) {
        const int idx = tid + s * NT;
        if (idx < ITEMS) {
            const int lp = idx & (kPkPairs - 1), b = idx >> 3;
            const int k = b % P;
            const int o0 = (b - k) * R + k;
#pragma unroll
            for (int q = 0; q < R; ++q) pk_sts<N>(buf, o0 + q * P, lp, u[s][q]);
        }
    }
#else
    // emulation (one thread): same two phases over a scratch copy of the tile
    (void)tid; (void)nt;
    cpk *all = new cpk[(size_t)ITEMS * R];
    for (int idx = 0; idx < ITEMS; ++idx) {
        const int lp = idx & (kPkPairs - 1), b = idx >> 3;
        const int k = b % P;
        cpk u[R];
        for (int r = 0; r < R; ++r) u[r] = pk_lds<N>(buf, b + r * T, lp);
        c64 pw[R];
        for (int r = 1; r < R; ++r) pw[r] = c.tw[r * k * STEP];
        for (int r = 1; r < R; ++r) u[r] = k_mul_w(u[r], pw[r]);
        DftK<R>::run(u);
        for (int r = 0; r < R; ++r) all[(size_t)idx * R + r] = u[r];
    }
    for (int idx = 0; idx < ITEMS; ++idx) {
        const int lp = idx & (kPkPairs - 1), b = idx >> 3;
        const int k = b % P;
        const int o0 = (b - k) * R + k;
        for (int q = 0; q < R; ++q) pk_sts<N>(buf, o0 + q * P, lp, all[(size_t)idx * R + q]);
    }
    delete[] all;
#endif
}

// Tiles the window mechanism lets a pass skip: forward passes skip tiles whose output window is empty;
// inverse passes replace tiles whose input window is empty by zeros in the output window.  Returns
// true when `tile` needs the transform.
IB_HD bool pkp_tile_active(const IlPassArgs &a, int64_t tile) {
    if (!a.win || a.win_mode == 0) return true;
    int lo, hi;
    pkp_tile_window(a, tile, a.win_mode == 2, lo, hi);
    return hi > lo;
}
IB_HD void pkp_tile_zero_fill(const IlPassArgs &a, int64_t tile, int tid, int nt) {
    c64 *g = const_cast<c64 *>(pkp_tile_base(a, tile));
    const int chunks = (a.out1 - a.out0) * kPkPairs;
    for (int i = tid; i < chunks; i += nt) {
        const int pos = a.out0 + (i >> 3), ch = i & 7;
        c64 *dst = g + (uint64_t)(unsigned)pos * a.pstride + 2 * ch;
        dst[0] = h_mk(0.f, 0.f); dst[1] = h_mk(0.f, 0.f);
    }
}
// first tile >= t (stride `step`) that needs the transform; inactive tiles of an inverse pass are
// zero-filled on the way.  Returns -1 when none is left.
IB_HD int64_t pkp_next_active(const IlPassArgs &a, int64_t t, int64_t step, int64_t ntiles, int tid, int nt) {
    for (; t < ntiles; t += step) {
        if (pkp_tile_active(a, t)) return t;
        if (a.win_mode == 2) pkp_tile_zero_fill(a, t, tid, nt);
    }
    return -1;
}

// registers the in-place middle stage needs per thread (complex pairs); the persistent form is used
// when this stays within 16 (N <= 512 with the radices of IB200_FFT_SPEC_LIST)
IB_HD constexpr int pkp_mid_pairs(int n, int r1, int r2, int nt) { return r2 > 1 ? ((kSpecL / 2 * (n / r1) + nt - 1) / nt) * r1 : 0; }

// one tile whose input already sits in raw[]; prefetches `next` (< 0: none) once raw[] is free.
// NT = threads of the CTA (0 in the single-threaded emulation)
template <int N, int R0, int R1, int R2, bool SWAP_IN, bool SWAP_OUT, int NT>
IB_HD void fft_pkp_tile_body(const IlPassArgs &a, int64_t tile, int64_t next, float *bufA, c64 *raw, int tid, int nt,
                             const c64 *tw = nullptr) {
    constexpr bool THREE = R2 > 1;
    PkPrefCtx<SWAP_IN, SWAP_OUT> c;
    c.raw = raw; c.gout = const_cast<c64 *>(pkp_tile_base(a, tile)); c.tw = tw ? tw : a.tw; c.pstride = a.pstride;
    int lo, hi;
    pkp_tile_window(a, tile, true, lo, hi);
    c.in0 = lo; c.inlen = (unsigned)(hi - lo);
    pkp_tile_window(a, tile, false, lo, hi);
    c.out0 = lo; c.outlen = (unsigned)(hi - lo);
    pk_stage<N, R0, 1, true, false, NT>(c, nullptr, bufA, tid, nt);
    IB_SYNC();                                                       // raw[] consumed, bufA complete
    if (next >= 0) pkp_prefetch(a, next, raw, tid, nt);
    if (THREE) {
        pk_stage_inplace<N, R1, R0, NT>(c, bufA, tid, nt);
        IB_SYNC();
        pk_stage<N, THREE ? R2 : R1, R0 * R1, false, true, NT>(c, bufA, nullptr, tid, nt);
    } else {
        pk_stage<N, R1, R0, false, true, NT>(c, bufA, nullptr, tid, nt);
    }
}

// ---- Toeplitz convolution pass (fused Toeplitz normal operator) ------------------------------------
// One tile of the last transformed axis: forward transform of the input window, multiplication by the
// real kernel K, re/im swap, forward transform again, store of the output window.  The stored lines are
// the inverse transform in the swapped state the first inverse pass of ib200_sense_ifft_combine leaves
// (the later inverse passes run forward transforms on swapped data), because K is real and commutes with
// the conjugation.  K is indexed by position along the axis and grid point: kern[pos * kplane + (line of
// the slab) / C].  Shared memory is that of the persistent pass (bufA + raw[] + twiddles): raw[] serves as
// the second buffer of the stages, and the next tile is prefetched into it once the second transform has left
// it, under the last stage (no stage runs in place: in-place stages, which would let the prefetch start
// earlier, hold more registers than the 128 two CTAs per SM allow and spill).
template <int N, int R0, int R1, int R2, int NT>
IB_HD void fft_pkt_tile_body(const IlPassArgs &a, int64_t tile, int64_t next, float *bufA, c64 *raw, int tid, int nt,
                             const c64 *tw, const float *kern, int64_t kplane, int C) {
    constexpr bool THREE = R2 > 1;
    float *bufB = reinterpret_cast<float *>(raw);
    PkPrefCtx<false, false> c;
    c.raw = raw; c.gout = const_cast<c64 *>(pkp_tile_base(a, tile)); c.tw = tw; c.pstride = a.pstride;
    c.in0 = a.in0; c.inlen = (unsigned)(a.in1 - a.in0); c.out0 = a.out0; c.outlen = (unsigned)(a.out1 - a.out0);
    pk_stage<N, R0, 1, true, false, NT>(c, nullptr, bufA, tid, nt);
    IB_SYNC();                                                       // raw[] consumed, bufA complete
    pk_stage<N, R1, R0, false, false, NT>(c, bufA, bufB, tid, nt);
    IB_SYNC();
    float *spec = bufB;                                              // spectrum: bufB (two stages) or bufA (three)
    if (THREE) {
        pk_stage<N, THREE ? R2 : R1, R0 * R1, false, false, NT>(c, bufB, bufA, tid, nt);
        IB_SYNC();
        spec = bufA;
    }
    // spectrum * K, swapped; the two lines of a pair may belong to two grid points (odd coil counts)
    const unsigned s0 = (unsigned)((tile % (a.inner / kSpecL)) * kSpecL);     // a.inner < 2^32
#pragma unroll 8
    for (int i = tid; i < N * kPkPairs; i += (NT > 0 ? NT : nt)) {          // unrolled: the kernel loads overlap
        const int pos = i / kPkPairs, lp = i % kPkPairs;
        const unsigned p0 = (s0 + 2 * lp) / (unsigned)C, p1 = (s0 + 2 * lp + 1) / (unsigned)C;
        const float *kr = kern + (int64_t)pos * kplane;
#ifdef __CUDA_ARCH__
        const pk2 kv = p_make(__ldg(kr + p0), __ldg(kr + p1));
#else
        const pk2 kv = p_make(kr[p0], kr[p1]);
#endif
        const cpk v = pk_lds<N>(spec, pos, lp);
        pk_sts<N>(spec, pos, lp, k_mk(p_mul(v.y, kv), p_mul(v.x, kv)));
    }
    IB_SYNC();
    if (THREE) {
        pk_stage<N, R0, 1, false, false, NT>(c, bufA, bufB, tid, nt);
        IB_SYNC();
        pk_stage<N, R1, R0, false, false, NT>(c, bufB, bufA, tid, nt);
        IB_SYNC();                                                   // raw[] free again
        if (next >= 0) pkp_prefetch(a, next, raw, tid, nt);
        pk_stage<N, THREE ? R2 : R1, R0 * R1, false, true, NT>(c, bufA, nullptr, tid, nt);
    } else {
        pk_stage<N, R0, 1, false, false, NT>(c, bufB, bufA, tid, nt);
        IB_SYNC();                                                   // raw[] free again
        if (next >= 0) pkp_prefetch(a, next, raw, tid, nt);
        pk_stage<N, R1, R0, false, true, NT>(c, bufA, nullptr, tid, nt);
    }
}

// ---- x passes of the fused SENSE transforms ------------------------------------------------------
// Lines are coils (fft_il.cuh: sense_x_tile); a pair is two neighbouring coils of one image row, so
// the coil count must be even.
struct PkXCtx {
    const c64 *tw;
    int npairs;
    // geometry of the tile
    int lmask, lshift;                 // line l -> coil (l & lmask), row (l >> lshift)
    int C, N0, off0;
    int64_t rowstride;                 // grid elements between neighbouring image rows (n0 * C)
    // expand: image and pf of the first voxel of the tile, grid row of the tile (+ coil chunk)
    const c64 *img, *pf;
    c64 *grow;
    int c0;
    IB_HD cpk gload(int lp, int pos) const {      // zpad(img * pf) at grid position pos
        const int j = pos - off0;
        if ((unsigned)j >= (unsigned)N0) return k_zero();
        const int l = 2 * lp;
        const int64_t vox = (int64_t)(l >> lshift) * N0 + j;
        const c64 iv = img[vox];
        const PkQuad q = pk_gld(pf + vox * C + c0 + (l & lmask));
        return k_mul_w(pk_from_f4(q.r0, q.i0, q.r1, q.i1), iv);
    }
    IB_HD void gstore(int lp, int pos, cpk v) const {
        const int l = 2 * lp;
        pk_gst(grow + (int64_t)(l >> lshift) * rowstride + (int64_t)pos * C + (l & lmask), v);
    }
};

template <int N, int R0, int R1, int R2, int NT>
IB_HD void sense_expand_pk_body(const SenseFftArgs &a, float *bufA, int64_t block, int tid, int nt,
                                const c64 *tw = nullptr) {
    const XTile t = sense_x_tile(a.C);
    const int ygroups = (a.N1 + t.YY - 1) / t.YY;
    const int y = (int)(block % ygroups) * t.YY, z = (int)(block / ygroups);
    const int rows = a.N1 - y < t.YY ? a.N1 - y : t.YY;
    const int64_t vox0 = ((int64_t)z * a.N1 + y) * a.N0;
    PkXCtx c;
    c.tw = tw ? tw : a.tw; c.C = a.C; c.N0 = a.N0; c.off0 = a.off0;
    c.lmask = t.YY > 1 ? t.CT - 1 : 0x7fffffff; c.lshift = t.YY > 1 ? t.shift : 31;
    c.rowstride = (int64_t)a.n0 * a.C;
    c.img = a.img + vox0; c.pf = a.pf + vox0 * a.C;
    const int64_t row = ((int64_t)(z + a.off2) * a.n1 + (y + a.off1)) * (int64_t)a.n0 * a.C;
    for (int c0 = 0; c0 < a.C; c0 += kSpecL) {
        const int nl = t.YY > 1 ? rows * t.CT : (a.C - c0 < kSpecL ? a.C - c0 : kSpecL);
        c.npairs = nl / 2; c.c0 = c0; c.grow = a.grid + row + c0;
        pk_run_stages<N, R0, R1, R2, false, NT>(c, bufA, tid, nt);
        IB_SYNC();
    }
}

// inverse x pass + coil combination (see sense_combine_body).  The last stage hands every cropped
// position to gstore(), which swaps re/im back (the inverse transform ran on swapped data),
// multiplies by conj(pf) -- two coils of one voxel are 16 contiguous bytes of pf -- and leaves the
// products in shared memory; one thread per (row, position) then folds the coils with 8-byte reads
// whose pair order is rotated by the position so that a warp spreads over the banks.
struct PkXInCtx {
    const c64 *tw;
    int npairs;
    int lmask, lshift, C;
    int64_t rowstride;
    const c64 *grow;
    // epilogue of the last stage
    float *res;                        // split planes res[j*16 + l], im plane NPOS*16 floats further
    int resplane;                      // floats between the planes
    const c64 *pf;                     // pf of the first voxel of the tile, + coil chunk
    int N0, off0;
    IB_HD cpk gload(int lp, int pos) const {
        const int l = 2 * lp;
        const PkQuad q = pk_gld(grow + (int64_t)(l >> lshift) * rowstride + (int64_t)pos * C + (l & lmask));
        return pk_from_f4(q.r0, q.i0, q.r1, q.i1);
    }
    IB_HD void gstore(int lp, int pos, cpk u) const {
        const int j = pos - off0;
        if ((unsigned)j >= (unsigned)N0) return;
        const int l = 2 * lp;
        const PkQuad q = pk_gld(pf + ((int64_t)(l >> lshift) * N0 + j) * C + (l & lmask));
        const pk2 px = p_make(q.r0, q.r1), py = p_make(q.i0, q.i1);
        // (im + i re) * conj(px + i py) = (im*px + re*py) + i (re*px - im*py)
        const pk2 ox = p_fma(u.y, px, p_mul(u.x, py));
        const pk2 oy = p_sub(p_mul(u.x, px), p_mul(u.y, py));
        reinterpret_cast<pk2 *>(res + j * kSpecL)[lp] = ox;
        reinterpret_cast<pk2 *>(res + resplane + j * kSpecL)[lp] = oy;
    }
};

template <int N, int R0, int R1, int R2, int NT>
IB_HD void sense_combine_pk_body(const SenseFftArgs &a, float *bufA, c64 *acc, int64_t block, int tid, int nt,
                                 const c64 *tw = nullptr) {
    constexpr bool THREE = R2 > 1;
    const XTile t = sense_x_tile(a.C);
    const int ygroups = (a.N1 + t.YY - 1) / t.YY;
    const int y = (int)(block % ygroups) * t.YY, z = (int)(block / ygroups);
    const int rows = a.N1 - y < t.YY ? a.N1 - y : t.YY;
    const int64_t vox0 = ((int64_t)z * a.N1 + y) * a.N0;
    float *bufB = bufA + pk_buf_floats(N);
    PkXInCtx c;
    c.tw = tw ? tw : a.tw; c.C = a.C; c.N0 = a.N0; c.off0 = a.off0;
    c.lmask = t.YY > 1 ? t.CT - 1 : 0x7fffffff; c.lshift = t.YY > 1 ? t.shift : 31;
    c.rowstride = (int64_t)a.n0 * a.C;
    c.resplane = N * kSpecL;
    const int64_t row = ((int64_t)(z + a.off2) * a.n1 + (y + a.off1)) * (int64_t)a.n0 * a.C;
    for (int c0 = 0; c0 < a.C; c0 += kSpecL) {
        const int nl = t.YY > 1 ? rows * t.CT : (a.C - c0 < kSpecL ? a.C - c0 : kSpecL);
        const int ncl = t.YY > 1 ? t.CT : nl;                       // coils of one row in this tile (even)
        c.npairs = nl / 2; c.grow = a.grid + row + c0; c.pf = a.pf + vox0 * a.C + c0;
        pk_stage<N, R0, 1, true, false, NT>(c, nullptr, bufA, tid, nt);
        IB_SYNC();
        if (THREE) {
            pk_stage<N, R1, R0, false, false, NT>(c, bufA, bufB, tid, nt);
            IB_SYNC();
            c.res = bufA;
            pk_stage<N, THREE ? R2 : R1, R0 * R1, false, true, NT>(c, bufB, nullptr, tid, nt);
        } else {
            c.res = bufB;
            pk_stage<N, R1, R0, false, true, NT>(c, bufA, nullptr, tid, nt);
        }
        IB_SYNC();
        const float *re = c.res, *im = c.res + c.resplane;
        const int np = ncl / 2;
        const bool single = a.C <= kSpecL;                         // one coil chunk: the fold goes straight to the image
        for (int i = tid; i < rows * a.N0; i += nt) {
            const int yy = i / a.N0, j = i - yy * a.N0;
            const float *pr = re + j * kSpecL + yy * ncl, *pi = im + j * kSpecL + yy * ncl;
            float sx = 0.f, sy = 0.f;
            int p = (j >> 1) % np;
            for (int q = 0; q < np; ++q) {
                sx += pr[2 * p] + pr[2 * p + 1];
                sy += pi[2 * p] + pi[2 * p + 1];
                if (++p == np) p = 0;
            }
            if (single) {
                c64 v = h_mul(a.alpha, h_mk(sx, sy));
                if (!a.beta_zero) v = h_add(v, h_mul(a.beta, a.img_out[vox0 + i]));
                a.img_out[vox0 + i] = v;
            } else {
                acc[i] = c0 == 0 ? h_mk(sx, sy) : h_add(acc[i], h_mk(sx, sy));
            }
        }
        IB_SYNC();
    }
    if (a.C <= kSpecL) return;
    for (int i = tid; i < rows * a.N0; i += nt) {
        c64 v = h_mul(a.alpha, acc[i]);
        if (!a.beta_zero) v = h_add(v, h_mul(a.beta, a.img_out[vox0 + i]));
        a.img_out[vox0 + i] = v;
    }
}

}  // namespace ib200
