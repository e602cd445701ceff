// Stage 1 (Tukey slicing + slice FFT), stage 3b (plane sum + slice IFFT) and stage 4 (50 % overlap-add)
// of the sliCQT path.  One CTA per (row, slice) unit; the whole length-L real transform lives in shared memory.
//
// The length-L real slice transform (L = 18060 for the pretrained Bark parameters) runs as ONE complex FFT of
// length N = L/2 = 9030 = 43 * 15 * 14 with the Good-Thomas prime-factor algorithm: the factors are pairwise
// coprime, so there are NO twiddle multiplications between the passes.  Round 2 design ("natural-order PFA"):
// the index permutations of the algorithm are folded into the first and the last pass, so that there is no
// separate permuting load / store phase and no per-element index arithmetic anywhere:
//
//   Ruritanian side  index = (210 i1 + 43 m) mod N, m = (14 i2 + 15 i3) mod 210.  A thread of pass A owns the
//                    column m (lanes <-> consecutive m: stride 43 words, conflict free) and finds its 43
//                    elements in NATURAL order at 43 m + 210 i1, minus N from the wrap point on (one select).
//   CRT side         (i1, i2, i3) = (index mod 43, mod 15, mod 14).  A thread of pass C owns the orbit
//                    {t + 645 j} of the last axis (lanes <-> consecutive t: coalesced global access); element j
//                    of the orbit has i3 = (t + j) mod 14, a rotation that costs one select per element.
//
//   analysis   x (global, CRT side) -> pass C (Tukey window on load, DFT-14) -> pass B (DFT-15) -> pass A (DFT-43)
//              -> natural order in shared memory -> even/odd split -> padded half spectrum H (global)
//   synthesis  two bin planes of T (global) summed in natural order -> Hermitian pre-processing -> pass A -> pass B
//              -> pass C, whose outputs go straight to y (store for even slices, red.add for odd slices)
//
// Pass A is the 43-point symmetric direct form streamed over the inputs and split BY OUTPUTS over two threads per
// column (Dftp<43, 2>, gen_codelets.py): 22 complex accumulators per thread, all twiddles immediates, and every
// operation one packed FFMA2 / FADD2.  Passes B and C are the packed straight-line codelets dft<15> / dft<14>.
//
// reference: nsgt/slicing.py:7-72 + nsgt/nsgtf.py:40 (forward), nsgt/nsigtf.py:93-103 +
//            nsgt/unslicing.py:33-69 + nsgt/slicq.py:207-230 (inverse); closed forms in DESIGN.md.
#include "slicq_common.cuh"
#include "dft_codelets.cuh"

namespace {

constexpr int kSliceThreads = 448;
// CTAs ahead whose input a CTA asks L2 to fetch while it transforms its own (synthesis: kPrefetchAhead, analysis:
// kPrefetchFwd).  Swept on the synthesis kernel:
// 32 / 64 / 96 / 128 / 148 / 208 / 296 / 592 CTAs ahead = 0.520 / 0.505 / 0.506 / 0.511 / 0.512 / 0.521 / 0.545 / 0.620 ms (off: 0.545;
// 296 CTAs are resident: further ahead the lines are evicted again before they are used)
constexpr int kPrefetchAhead = 80;
constexpr int kPrefetchFwd = 80;

constexpr int cmodinv(int a, int m) {
    a %= m;
    for (int x = 1; x < m; ++x)
        if ((a * x) % m == 1) return x;
    return 0;
}

template <int P1_, int P2_, int P3_, int NP_, int SB_, int SA_>
struct PfaNat {
    static constexpr int P1 = P1_, P2 = P2_, P3 = P3_, NP = NP_;
    static constexpr int N = P1 * P2 * P3, Q = P2 * P3, C3 = N / P3;
    static constexpr int SB = SB_, SA = SA_;                 // pitches of the (i1, i2, i3) layout between the passes
    static constexpr int SLOT = (Q + 31) / 32 * 32;          // pass A: threads per part (warp multiple >= Q)
    // Natural order as pass C sees it: row k = n / C3 of the natural index n starts at k * PN.  Lane t of pass C touches
    // t + PN * ((c - t) mod P3): with PN a multiple of 16 words the bank depends on t alone (conflict free); with the
    // plain pitch C3 = 645 the lanes of a half warp fall on 4 banks.
    static constexpr int PN = (C3 + 15) / 16 * 16;
    SLICQ_DEVFN static int natp(int n) { return n + (PN - C3) * (n / C3); }
    static constexpr int SMEM_A_ = (P1 * SA > N + 2 ? P1 * SA : N + 2);
    static constexpr int SMEM_ELEMS = (SMEM_A_ > P3 * PN ? SMEM_A_ : P3 * PN);
    static constexpr int I2 = cmodinv(P3, P2), I3 = cmodinv(P2, P3);   // m -> (i2, i3) = (I2 m mod P2, I3 m mod P3)
    static_assert(C3 % P3 == 1, "orbit rotation of the last axis assumes (N / P3) mod P3 == 1");
    static_assert(SA >= P2 * SB && SB >= P3, "pitches too small");
    static_assert(NP * SLOT <= kSliceThreads, "pass A needs NP * SLOT threads");
};
typedef PfaNat<43, 15, 14, 2, 16, 243> Pfa9030;

// pass A sources / destinations (Dftp<>::run / store)
template <class PF> struct ColNat {        // column m in natural order: element i1 at 43 m + 210 i1 (mod N)
    float2* lo; float2* hi; int nw;
    SLICQ_DEVFN ColNat(float2* Z, int m) {
        lo = Z + PF::P1 * m;
        hi = lo - PF::N;
        nw = (PF::N - PF::P1 * m + PF::Q - 1) / PF::Q;       // first i1 past the wrap
    }
    SLICQ_DEVFN cpx ld(int i) const { return cpx_ld((i >= nw ? hi : lo) + PF::Q * i); }
    SLICQ_DEVFN void st(int i, cpx v) const { cpx_st((i >= nw ? hi : lo) + PF::Q * i, v); }
};
template <class PF> struct ColL2 {         // column (i2, i3) of the pitched layout: element i1 at i1 * SA + i2 * SB + i3
    float2* p;
    SLICQ_DEVFN ColL2(float2* Z, int m) { p = Z + ((PF::I2 * m) % PF::P2) * PF::SB + ((PF::I3 * m) % PF::P3); }
    SLICQ_DEVFN cpx ld(int i) const { return cpx_ld(p + PF::SA * i); }
    SLICQ_DEVFN void st(int i, cpx v) const { cpx_st(p + PF::SA * i, v); }
};

// pass A: DFT-P1 of every column; SRC / DST = the layout the pass reads / writes (both alias Z: all reads
// complete before the first write)
template <class PF, bool INV, class SRC, class DST>
SLICQ_DEVFN void pass_a(float2* Z) {
    typedef Dftp<PF::P1, PF::NP, INV> D;
    const int part = threadIdx.x / PF::SLOT, m = threadIdx.x - part * PF::SLOT;
    const bool act = part < PF::NP && m < PF::Q;
    cpx o[D::NOUT];
    if (act) { SRC s(Z, m); D::run(part, s, o); }
    __syncthreads();
    if (act) { DST d(Z, m); D::store(part, d, o); }
    __syncthreads();
}

// pass B: DFT-P2 along i2 for fixed (i1, i3), in place; lanes <-> i1 (pitch SA odd: conflict free)
template <class PF, bool INV>
SLICQ_DEVFN void pass_b(float2* Z) {
    for (int t = threadIdx.x; t < PF::P1 * PF::P3; t += kSliceThreads) {
        const int i3 = t / PF::P1, i1 = t - i3 * PF::P1;
        float2* p = Z + i1 * PF::SA + i3;
        cpx v[PF::P2];
#pragma unroll
        for (int b = 0; b < PF::P2; ++b) v[b] = cpx_ld(p + b * PF::SB);
        dft<PF::P2, INV>(v);
#pragma unroll
        for (int b = 0; b < PF::P2; ++b) cpx_st(p + b * PF::SB, v[b]);
    }
    __syncthreads();
}

}  // namespace

// ------------------------------------------------------------------------------------------
// stage 1: one CTA per (row, slice).  x -> padded half spectrum H_ext[pad_l + f], f in [-pad_l, N + pad_r]
template <class PF>
__global__ void __launch_bounds__(kSliceThreads, 2) slice_fft_fwd_kernel(const __grid_constant__ SlicqSliceParams p) {
    SLICQ_DYN_SMEM(float2, Z);
    constexpr int N = PF::N, NT = kSliceThreads, P3 = PF::P3, C3 = PF::C3;
    const int rsl = blockIdx.x;
    const int rs = p.rs0 + rsl;
    const int row = rs / p.S, k = rs - row * p.S;
    const long long s0 = (p.k0 + k - 1) * (long long)p.t.hop - p.t0;  // x index of slice sample 0
    const float* __restrict__ xr = p.x + row * p.x_row_stride;
    const float2* __restrict__ tw2 = reinterpret_cast<const float2*>(p.t.tukey);
    const int e_lo = p.t.tw_lo >> 1, e_hi = (p.t.tw_hi + 1) >> 1;       // sample pairs with a non-zero window
    const long long sa = s0 + 2 * e_lo, sb = s0 + 2 * e_hi;             // x range touched by the window support
    const bool fast = sa >= 0 && sb <= p.T && ((reinterpret_cast<uintptr_t>(xr + s0) & 7) == 0);
    if (blockIdx.x + kPrefetchFwd < gridDim.x) {
        // the second half of the slice kPrefetchFwd units ahead (its first half is the second half of its left neighbour)
        const int rs2 = rs + kPrefetchFwd;
        const int row2 = rs2 / p.S, k2 = rs2 - row2 * p.S;
        const long long a = (p.k0 + k2) * (long long)p.t.hop - p.t0;          // x index of the middle of that slice
        const float* __restrict__ x2r = p.x + row2 * p.x_row_stride;
        for (long long i = a + 32LL * threadIdx.x; i < a + p.t.hop; i += 32LL * NT)
            if (i >= 0 && i < p.T) prefetch_l2(x2r + i);
    }
    // ---- windowed slice -> Z in natural order (coalesced loads; the zero part of the window is not read)
    if (fast) {
        const float2* __restrict__ x2 = reinterpret_cast<const float2*>(xr + s0);
        constexpr int U = 5;
        for (int e0 = threadIdx.x; e0 < N; e0 += U * NT) {
            float2 xv[U], wv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int e = e0 + u * NT;
                if (e >= e_lo && e < e_hi) { xv[u] = __ldg(x2 + e); wv[u] = __ldg(tw2 + e); }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int e = e0 + u * NT;
                if (e < N) Z[PF::natp(e)] = (e >= e_lo && e < e_hi) ? make_float2(xv[u].x * wv[u].x, xv[u].y * wv[u].y) : make_float2(0.f, 0.f);
            }
        }
    } else {
        for (int e = threadIdx.x; e < N; e += NT) {
            const long long sx = s0 + 2 * e;
            const float2 wv = __ldg(tw2 + e);
            float a = 0.f, b = 0.f;
            if (sx >= 0 && sx < p.T) a = __ldg(xr + sx) * wv.x;
            if (sx + 1 >= 0 && sx + 1 < p.T) b = __ldg(xr + sx + 1) * wv.y;
            Z[PF::natp(e)] = make_float2(a, b);
        }
    }
    __syncthreads();
    // ---- pass C (first): thread t owns the orbit {t + C3 j} of the natural order; element j has i3 = (t + j) mod P3.
    // The outputs go to the pitched layout, which aliases the natural one: all tasks of a thread stay in registers
    // until every thread has read its inputs.
    {
        constexpr int NRC = (C3 + NT - 1) / NT;
        cpx v[NRC][P3];
#pragma unroll
        for (int r = 0; r < NRC; ++r) {
            const int t = threadIdx.x + r * NT;
            if (t < C3) {
                const int s = t % P3;
                const int j0 = s ? P3 - s : 0, w = P3 - j0;      // v[c] = element j0 + c (mod P3); wraps for c >= w
                const float2* za = Z + t + j0 * PF::PN;
                const float2* zb = za - P3 * PF::PN;
#pragma unroll
                for (int c = 0; c < P3; ++c) v[r][c] = cpx_ld((c >= w ? zb : za) + c * PF::PN);
                dft<P3, false>(v[r]);
            }
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < NRC; ++r) {
            const int t = threadIdx.x + r * NT;
            if (t < C3) {
                float2* o = Z + (t % PF::P1) * PF::SA + (t % PF::P2) * PF::SB;
#pragma unroll
                for (int c = 0; c < P3; ++c) cpx_st(o + c, v[r][c]);
            }
        }
    }
    __syncthreads();
    pass_b<PF, false>(Z);
    pass_a<PF, false, ColL2<PF>, ColNat<PF> >(Z);
    // ---- even/odd split: H[k] = E + w^k O, H[N-k] = conj(E - w^k O); mirrored margins for the bins
    // that reach below DC / above Nyquist (Hermitian symmetry of a real slice)
    float2* __restrict__ H = p.spec + (long long)rsl * p.spec_stride + p.t.pad_l;
    const int pad_l = p.t.pad_l, pad_r = p.t.pad_r;
    const float sc = 0.5f * p.t.spec_scale, se = p.t.ends_scale;
    const float mir = (p.t.adjoint & 1) ? 0.f : 1.f;     // adjoint mode: positions outside [0, N] read as zero
    constexpr int NP2 = (N / 2 + NT) / NT;      // pairs (k, N-k) per thread
    float2 wkv[NP2];
#pragma unroll
    for (int u = 0; u < NP2; ++u) {
        const int kk = threadIdx.x + u * NT;
        if (kk <= N / 2) wkv[u] = __ldg(p.t.post_tw + kk);
    }
#pragma unroll
    for (int u = 0; u < NP2; ++u) {
        const int kk = threadIdx.x + u * NT;
        if (kk > N / 2) continue;
        const cpx zk = cpx_ld(Z + kk);
        if (kk == 0) {
            const float a = cpx_re(zk), b = cpx_im(zk);
            H[0] = make_float2((a + b) * se, 0.f);
            H[N] = make_float2((a - b) * se, 0.f);
        } else {
            const cpx zn = cpx_ld(Z + N - kk);
            const float2 wk = wkv[u];
            const cpx E = caddc(zk, zn);                    // zk + conj(zn)           (= 2 E)
            const cpx D = csubc(zk, zn);                    // zk - conj(zn)           (= 2 i O)
            const cpx t = cmulw(D, wk);                     // w^k (zk - conj zn) = 2 i w^k O
            // H[k] = E + w^k O = (2E - i t) / 2 ; H[N-k] = conj(E - w^k O) = conj(2E + i t) / 2
            const cpx hk = cmulr(csubi(E, t), sc);
            const cpx hn = cmulr(cconjp(caddi(E, t)), sc);
            cpx_st(H + kk, hk);
            cpx_st(H + N - kk, hn);
            if (kk <= pad_l) cpx_st(H - kk, cmulr(cconjp(hk), mir));
            if (kk <= pad_r) cpx_st(H + N + kk, cmulr(cconjp(hn), mir));
        }
    }
}

// ------------------------------------------------------------------------------------------
// stage 3b + 4: one CTA per (row, slice).  T row = two planes of windowed bin spectra (even bins / odd bins at
// their spectrum positions, written by bins_inv_kernel) + a short overflow list for the few positions where two
// bins of one plane overlap.  u = IRFFT(plane 0 + plane 1 + overflow), overlap-added straight into y:
// y[(k-1)*hop + p] += u_k[p].  Every output sample is the sum of exactly two slices, one even and one odd: the
// launch with parity 0 STORES the even slices, the launch with parity 1 (stream-ordered after it) ADDS the odd ones
// with fire-and-forget reductions (red.global.add: every location receives exactly one addition, so no ordering
// question arises) -- no intermediate slice buffer, and a two-term sum is order independent (bitwise reproducible).
// (reference: nsgt/nsigtf.py:82-103, nsgt/unslicing.py:33-69, nsgt/slicq.py:207-230)
template <class PF>
__global__ void __launch_bounds__(kSliceThreads, 2) slice_fft_inv_kernel(const __grid_constant__ SlicqSliceParams p) {
    SLICQ_DYN_SMEM(float2, Z);
    constexpr int N = PF::N, NT = kSliceThreads, P3 = PF::P3, C3 = PF::C3;
    // CTA i of the launch = i-th slice of this launch's parity at or after unit rs0
    const int pi = p.par_base + blockIdx.x;
    const int row = pi / p.par_cs, k = 2 * (pi - row * p.par_cs) + p.parity;
    const int rsl = row * p.S + k - p.rs0;
    const int tid = threadIdx.x;
    const float2* __restrict__ Trow = p.spec + (long long)rsl * p.spec_stride;
    // ---- R[f] = plane0[f] + plane1[f] (+ overflow), f in [0, N], and the Hermitian pre-processing, with ONE memory round
    // trip and one pass over shared memory.  Plane 0 lands in Z by bulk copy (TMA engine: no registers, no load/store
    // pipe traffic); meanwhile every thread loads plane 1 at ITS pairs (k, N - k) into registers.  After the copy has
    // landed (mbarrier) and the overflow entries are added, a thread owns its pairs exclusively: it adds plane 1,
    // pre-processes and writes back in place.
    constexpr int NP2 = (N / 2 + NT) / NT;      // pairs (k, N-k) per thread
    constexpr unsigned ROW_BYTES = (N / 2 + 1) * 16u;   // positions 0 .. N and one pad, rows are 16-byte aligned
#ifdef SLICQ_EMU
    unsigned long long bar_[1];
#else
    __shared__ __align__(8) unsigned long long bar_[1];
#endif
    if (tid == 0) mbar_init(bar_, 1);
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(bar_, ROW_BYTES);
        const unsigned char* src = reinterpret_cast<const unsigned char*>(Trow + p.t.pl_off);
        unsigned char* dst = reinterpret_cast<unsigned char*>(Z);
        constexpr unsigned PIECE = 9040;        // a few copies in flight instead of one long one
        for (unsigned o = 0; o < ROW_BYTES; o += PIECE)
            bulk_g2s(dst + o, src + o, (ROW_BYTES - o < PIECE) ? ROW_BYTES - o : PIECE, bar_);
    }
    {
        const float2* __restrict__ P1 = Trow + p.t.pl_off + p.t.pl_len;
        float2 b0[NP2], b1[NP2];
#pragma unroll
        for (int u = 0; u < NP2; ++u) {
            const int kk = tid + u * NT;
            if (kk <= N / 2) { b0[u] = __ldg(P1 + kk); b1[u] = __ldg(P1 + N - kk); }
        }
        int4 xe = make_int4(-1, 0, -1, 0);
        if (tid < p.t.n_ex) xe = __ldg(p.t.ex + tid);
        float2 x2 = make_float2(0.f, 0.f), x3 = make_float2(0.f, 0.f);
        if (xe.x >= 0) { x2 = __ldg(Trow + xe.y); if (xe.z >= 0) x3 = __ldg(Trow + xe.z); }
        {   // while this CTA transforms, L2 fetches the row of the CTA that will run in this slot next (blockIdx + resident CTAs)
            const int pj = pi + kPrefetchAhead;
            if (blockIdx.x + kPrefetchAhead < gridDim.x) {
                const int row2 = pj / p.par_cs, k2 = 2 * (pj - row2 * p.par_cs) + p.parity;
                const float2* __restrict__ T2 = p.spec + (long long)(row2 * p.S + k2 - p.rs0) * p.spec_stride;
                if (tid == 32) bulk_prefetch_l2(T2, (unsigned)p.t.t_stride * 8u);      // rows are 16-byte aligned, t_stride is even
            }
        }
        mbar_wait(bar_, 0);
        // overflow entries: position f also receives T[off0] (+ T[off1]); entries have distinct f
        if (xe.x >= 0) { Z[xe.x].x += x2.x + x3.x; Z[xe.x].y += x2.y + x3.y; }
        for (int i = tid + NT; i < p.t.n_ex; i += NT) {
            const int4 q = __ldg(p.t.ex + i);
            float2 e = __ldg(Trow + q.y);
            if (q.z >= 0) { const float2 v = __ldg(Trow + q.z); e.x += v.x; e.y += v.y; }
            Z[q.x].x += e.x; Z[q.x].y += e.y;
        }
        if (p.t.adjoint & 2) {
            // adjoint of the analysis: what the bins put below DC / above Nyquist folds back conjugated (the analysis
            // READS the Hermitian mirror there); positions 1 .. pad_l and N - pad_r .. N - 1, disjoint from the entries above
            // only in time: order them after the overflow pass
            __syncthreads();
            const float2* __restrict__ P0 = Trow + p.t.pl_off;
            for (int f = 1 + tid; f <= p.t.pad_l; f += NT) {
                const float2 a = __ldg(P0 - f), b = __ldg(P1 - f);
                Z[f].x += a.x + b.x; Z[f].y -= a.y + b.y;
            }
            for (int f = 1 + tid; f <= p.t.pad_r; f += NT) {
                const float2 a = __ldg(P0 + N + f), b = __ldg(P1 + N + f);
                Z[N - f].x += a.x + b.x; Z[N - f].y -= a.y + b.y;
            }
        }
        __syncthreads();
        // ---- plane sum + Hermitian pre-processing, in place: Z[k] = E + i conj(w^k) O, Z[N-k] = conj(E - i conj(w^k) O)
#pragma unroll
        for (int u = 0; u < NP2; ++u) {
            const int kk = tid + u * NT;
            if (kk > N / 2) continue;
            const float2 wk = __ldg(p.t.post_tw + kk);
            const cpx rk = cadd(cpx_ld(Z + kk), cpx_from(b0[u]));
            const cpx rn = cadd(cpx_ld(Z + N - kk), cpx_from(b1[u]));
            if (kk == 0) {
                // imaginary parts of DC / Nyquist are ignored by a C2R transform (nsigtf.py:103)
                const float es = (p.t.adjoint & 2) ? 2.f : 1.f;     // adjoint of the analysis: DC / Nyquist count twice
                const float a = cpx_re(rk) * es, b = cpx_re(rn) * es;
                Z[0] = make_float2(a + b, a - b);
            } else {
                const cpx E = caddc(rk, rn);                 // rk + conj(rn)
                const cpx O = csubc(rk, rn);                 // rk - conj(rn)
                const cpx t = cmulwc(O, wk);                 // conj(w^k) O
                cpx_st(Z + kk, caddi(E, t));                 // E + i t
                cpx_st(Z + N - kk, cconjp(csubi(E, t)));     // conj(E - i t)
            }
        }
    }
    __syncthreads();
    pass_a<PF, true, ColNat<PF>, ColL2<PF> >(Z);
    pass_b<PF, true>(Z);
    // ---- pass C (last): thread t owns the orbit {t + C3 j} of the OUTPUT; element j has i3 = (t + j) mod P3.  The
    // outputs go back to Z in natural order (all tasks of a thread stay in registers until every thread has read its
    // inputs) and leave as 14 bulk copies / bulk reductions (one per row of C3 = 645 sample pairs, issued by lane 0 of
    // warp j; TMA engine: no registers, no load/store pipe traffic) plus one ordinary access per row for the element that
    // the 16-byte alignment rule leaves over.  Row j of the staging area starts at Z + PN j + sh_j with sh_j in {0, 1}
    // chosen so that the 16-byte aligned part of the row in y is 16-byte aligned in shared memory as well (a row is
    // 5160 bytes: the alignment of its start in y alternates from row to row).
    // slice sample pair n = (2n, 2n+1) goes to y index tb + 2n;  first half (n < N/2) = hop k-1, second half = hop k
    static_assert(P3 % 2 == 0 && (P3 / 2) * C3 == N / 2 && NT / 32 >= P3, "row structure of the output staging");
    const long long tb = (p.k0 + k - 1) * (long long)p.t.hop - p.t0;
    float* __restrict__ yr = p.x + row * p.x_row_stride;
    const int q0 = (int)((reinterpret_cast<uintptr_t>(yr + tb) >> 3) & 1);       // 1: y + tb is 8 but not 16 bytes aligned
    {
        constexpr int NRC = (C3 + NT - 1) / NT;
        cpx v[NRC][P3];
#pragma unroll
        for (int r = 0; r < NRC; ++r) {
            const int t = tid + r * NT;
            if (t < C3) {
                const float2* src = Z + (t % PF::P1) * PF::SA + (t % PF::P2) * PF::SB;
#pragma unroll
                for (int c = 0; c < P3; ++c) v[r][c] = cpx_ld(src + c);
                dft<P3, true>(v[r]);
            }
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < NRC; ++r) {
            const int t = tid + r * NT;
            if (t < C3) {
                const int s = t % P3;
                const int j0 = s ? P3 - s : 0, w = P3 - j0;
                const int qq = (q0 + j0) & 1;                 // sh of the row of element c: qq for even c, 1 - qq for odd c
                float2* za0 = Z + t + j0 * PF::PN + qq;
                float2* za1 = Z + t + j0 * PF::PN + 1 - qq;
                float2* zb0 = za0 - P3 * PF::PN;
                float2* zb1 = za1 - P3 * PF::PN;
#pragma unroll
                for (int c = 0; c < P3; ++c) cpx_st((c >= w ? ((c & 1) ? zb1 : zb0) : ((c & 1) ? za1 : za0)) + c * PF::PN, v[r][c]);
            }
        }
    }
    auto stage = [&](int n) { const int j = n / C3; return n + (PF::PN - C3) * j + ((q0 + j) & 1); };   // natural index -> staging slot
    const bool accumulate = p.parity != 0;
    // the last slice of the call has no right neighbour: its second half is stored even when odd
    const bool second_store = !accumulate || (k + 1 >= p.S);
    const bool first_to_halo = (k == 0);      // hop -1: other shard (halo) or before the signal (dropped)
    float* __restrict__ halo = (p.halo_out != nullptr && p.k0 > 0) ? p.halo_out + (long long)row * p.t.hop : nullptr;
    const bool vec = ((reinterpret_cast<uintptr_t>(yr + tb) & 7) == 0) && tb >= 0 && tb + 2 * N <= p.T && !first_to_halo;
    const bool add1 = accumulate, add2 = accumulate && !second_store;
    if (p.t.adjoint & 2) {
        // adjoint of the analysis: the slicing window multiplies the slice before the overlap-add
        __syncthreads();
        const float2* __restrict__ tw2 = reinterpret_cast<const float2*>(p.t.tukey);
        for (int n = tid; n < N; n += NT) { const float2 w = __ldg(tw2 + n); float2& z = Z[stage(n)]; z.x *= w.x; z.y *= w.y; }
    }
    fence_proxy_async();
    __syncthreads();
    if (vec) {
        const int j = tid >> 5, lane = tid & 31;
        if (j < P3 && lane < 2) {
            const int sh = (q0 + j) & 1;
            const bool add = (j < P3 / 2) ? add1 : add2;
            float2* __restrict__ y2 = reinterpret_cast<float2*>(yr + tb) + C3 * j;
            float2* zr = Z + PF::PN * j + sh;                        // element e of the row at zr[e]
            if (lane == 0) {
                // elements sh .. sh + C3 - 2: 16-byte aligned on both sides
                if (add) bulk_s2g_add_f32(y2 + sh, zr + sh, (C3 - 1) * 8u); else bulk_s2g(y2 + sh, zr + sh, (C3 - 1) * 8u);
                bulk_wait_read();
            } else {
                const int e = sh ? 0 : C3 - 1;
                const float2 z = zr[e];
                if (add) slicq_red_add2(reinterpret_cast<float*>(y2 + e), z); else y2[e] = z;
            }
        }
    } else {
        for (int n = tid; n < N; n += NT) {
            const float2 z = Z[stage(n)];
            const bool first = n < N / 2;
            const bool add = first ? add1 : add2;
            if (first && first_to_halo) {
                if (halo) { halo[2 * n] = z.x; halo[2 * n + 1] = z.y; }
            } else {
                const long long ty = tb + 2 * n;
                if (ty >= 0 && ty < p.T) { if (add) slicq_red_add(yr + ty, z.x); else yr[ty] = z.x; }
                if (ty + 1 >= 0 && ty + 1 < p.T) { if (add) slicq_red_add(yr + ty + 1, z.y); else yr[ty + 1] = z.y; }
            }
        }
    }
}

// host-side helpers / launchers ---------------------------------------------------------------
extern "C" int slicq_generic_smem_bytes(int L);
extern "C" int slicq_launch_slice_fwd_generic(const SlicqSliceParams* p, cudaStream_t s);
extern "C" int slicq_launch_slice_inv_generic(const SlicqSliceParams* p, cudaStream_t s);

// shared memory of the slice kernels for slice length L: the tuned prime-factor kernels for the pretrained
// configuration, the generic kernels (k_slice_generic.cu) for every other length that fits; -1 = unsupported
extern "C" int slicq_slice_smem_bytes(int L) {
    if (L == 2 * Pfa9030::N) return (int)(Pfa9030::SMEM_ELEMS * sizeof(float2));
    return slicq_generic_smem_bytes(L);
}

extern "C" int slicq_launch_slice_fwd(const SlicqSliceParams* p, cudaStream_t s) {
    if (p->n_rs <= 0) return 0;
    if (p->t.L != 2 * Pfa9030::N) return slicq_launch_slice_fwd_generic(p, s);
    const int smem = (int)(Pfa9030::SMEM_ELEMS * sizeof(float2));
    if (slicq_smem_opt_in<slice_fft_fwd_kernel<Pfa9030>>(smem)) return -3;
    SLICQ_LAUNCH(slice_fft_fwd_kernel<Pfa9030>, dim3(p->n_rs), dim3(kSliceThreads), smem, s, *p);
    return (int)cudaGetLastError();
}

extern "C" int slicq_launch_slice_inv(const SlicqSliceParams* p, cudaStream_t s) {
    if (p->n_rs <= 0) return 0;
    if (p->t.L != 2 * Pfa9030::N) return slicq_launch_slice_inv_generic(p, s);
    const int smem = (int)(Pfa9030::SMEM_ELEMS * sizeof(float2));
    if (slicq_smem_opt_in<slice_fft_inv_kernel<Pfa9030>>(smem)) return -3;
    SlicqSliceParams sp;
    const unsigned ctas = slicq_parity_ctas(*p, sp);
    if (!ctas) return 0;
    SLICQ_LAUNCH(slice_fft_inv_kernel<Pfa9030>, dim3(ctas), dim3(kSliceThreads), smem, s, sp);
    return (int)cudaGetLastError();
}
