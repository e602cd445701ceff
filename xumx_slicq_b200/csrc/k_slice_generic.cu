// Generic slice kernels: any slice length L = 2 N the tuned prime-factor kernels (k_slice.cu, L = 18060) do not cover --
// other Bark / mel / log / linear configurations of the reference (SURVEY.md section 8(f) N4: nsgt/fscale.py:92-188,
// slicqfinder.py / optuna.py parameter searches).  Same stages, same data layout, same even/odd packing of the real
// transform; the length-N complex FFT is a Stockham autosort over the prime factors of N with direct radix-p butterflies
// (one output per thread and stage: O(N sum p) operations, any factor, natural order in and out; twiddles from one table
// exp(-2 pi i k / N)).  Correct for every N that fits two buffers in shared memory, not tuned: the roofline work is the
// pretrained configuration's.  Also here: the reference's mirrored-bin pass (nsgt/nsigtf.py:63-80) for configurations
// where a bin reaches below DC, so that its mirror image wraps into the kept half spectrum, and its transpose; and the
// transforms of the long Nyquist bin of band-limited filterbanks (fmax < fs / 2) on the same Stockham engine.
#include "slicq_common.cuh"

#define SLICQ_GEN_THREADS 256

namespace {

SLICQ_DEVFN float2 gmul(float2 a, float2 b) { return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x)); }

// x -> FFT (sign -) or unnormalised inverse FFT (sign +) of length N = prod fac[0 .. n_fac) (largest factor first);
// wN = exp(-2 pi i k / N), wP = exp(-2 pi i k / fac[0]) in double when fac[0] > 32.  Returns the buffer that holds the result
template <bool INV>
SLICQ_DEVFN float2* stockham(float2* x, float2* y, int N, int n_fac, const int* fac, const float2* wN, const double2* wP) {
    int n = N, s = 1;
    for (int st = 0; st < n_fac; ++st) {
        const int pf = fac[st], m = n / pf;
        const int wp = N / pf, wn = N / n;
        for (int idx = threadIdx.x; idx < N; idx += SLICQ_GEN_THREADS) {
            // output idx = r + s (pf q + j)  <-  inputs r + s (q + m k), k < pf
            const int r = idx % s, u = idx / s;
            const int j = u % pf, q = u / pf;
            const float2* src = x + r + s * q;
            float2 acc = src[0];
            int jk = 0;
            if (pf <= 32 || st != 0) {       // only the largest factor (first stage) has a double table
                for (int k = 1; k < pf; ++k) {
                    jk += j; if (jk >= pf) jk -= pf;
                    float2 w = __ldg(wN + wp * jk);
                    if (INV) w.y = -w.y;
                    const float2 a = src[s * m * k];
                    acc.x += a.x * w.x - a.y * w.y;
                    acc.y += a.x * w.y + a.y * w.x;
                }
            } else {
                // a large prime factor (e.g. 1721 for sl_len 6884) is a direct sum of pf terms: accumulate in double so that
                // the transform keeps the accuracy of an FFT (round-trip SNR within 0.1 dB of the reference)
                // (double twiddles too: fp32 twiddle rounding alone would add sqrt(pf) * 6e-8 of noise)
                double ax = acc.x, ay = acc.y;
                for (int k = 1; k < pf; ++k) {
                    jk += j; if (jk >= pf) jk -= pf;
                    double2 w = wP[jk];
                    if (INV) w.y = -w.y;
                    const float2 a = src[s * m * k];
                    ax += (double)a.x * w.x - (double)a.y * w.y;
                    ay += (double)a.x * w.y + (double)a.y * w.x;
                }
                acc = make_float2((float)ax, (float)ay);
            }
            float2 tw = __ldg(wN + wn * j * q);
            if (INV) tw.y = -tw.y;
            y[idx] = gmul(acc, tw);
        }
        __syncthreads();
        float2* tmp = x; x = y; y = tmp;
        n = m; s *= pf;
    }
    return x;
}

}  // namespace

__global__ void __launch_bounds__(SLICQ_GEN_THREADS, 1) slice_fft_fwd_generic_kernel(const __grid_constant__ SlicqSliceParams p) {
    SLICQ_DYN_SMEM(float2, A);
    const int N = p.t.N2, NT = SLICQ_GEN_THREADS;
    float2* B = A + N + 2;
    const int rsl = blockIdx.x;
    const int rs = p.rs0 + rsl;
    const int row = rs / p.S, k = rs - row * p.S;
    const long long s0 = (p.k0 + k - 1) * (long long)p.t.hop - p.t0;
    const float* __restrict__ xr = p.x + row * p.x_row_stride;
    const float2* __restrict__ tw2 = reinterpret_cast<const float2*>(p.t.tukey);
    for (int e = threadIdx.x; e < N; e += NT) {
        const long long sx = s0 + 2 * e;
        const float2 wv = __ldg(tw2 + e);
        float a = 0.f, b = 0.f;
        if (sx >= 0 && sx < p.T) a = __ldg(xr + sx) * wv.x;
        if (sx + 1 >= 0 && sx + 1 < p.T) b = __ldg(xr + sx + 1) * wv.y;
        A[e] = make_float2(a, b);
    }
    __syncthreads();
    const float2* Z = stockham<false>(A, B, N, p.t.n_fac, p.t.fac, p.t.wN, p.t.wP);
    float2* __restrict__ H = p.spec + (long long)rsl * p.spec_stride + p.t.pad_l;
    const int pad_l = p.t.pad_l, pad_r = p.t.pad_r;
    const float sc = p.t.spec_scale, se = p.t.ends_scale;
    const float mir = (p.t.adjoint & 1) ? 0.f : 1.f;
    for (int kk = threadIdx.x; kk <= N / 2; kk += NT) {
        const float2 zk = Z[kk];
        if (kk == 0) {
            H[0] = make_float2((zk.x + zk.y) * se, 0.f);
            H[N] = make_float2((zk.x - zk.y) * se, 0.f);
        } else {
            const float2 zn = Z[N - kk];
            const float2 wk = __ldg(p.t.post_tw + kk);
            const float2 E = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
            const float2 O = make_float2(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
            const float2 t = gmul(wk, O);
            const float2 hk = make_float2((E.x + t.x) * sc, (E.y + t.y) * sc);
            const float2 hn = make_float2((E.x - t.x) * sc, -(E.y - t.y) * sc);
            H[kk] = hk;
            H[N - kk] = hn;
            if (kk <= pad_l) H[-kk] = make_float2(hk.x * mir, -hk.y * mir);
            if (kk <= pad_r) H[N + kk] = make_float2(hn.x * mir, -hn.y * mir);
        }
    }
}

__global__ void __launch_bounds__(SLICQ_GEN_THREADS, 1) slice_fft_inv_generic_kernel(const __grid_constant__ SlicqSliceParams p) {
    SLICQ_DYN_SMEM(float2, A);
    const int N = p.t.N2, NT = SLICQ_GEN_THREADS;
    float2* B = A + N + 2;
    const int pi = p.par_base + blockIdx.x;
    const int row = pi / p.par_cs, k = 2 * (pi - row * p.par_cs) + p.parity;
    const int rsl = row * p.S + k - p.rs0;
    const int tid = threadIdx.x;
    const float2* __restrict__ Trow = p.spec + (long long)rsl * p.spec_stride;
    const float2* __restrict__ P0 = Trow + p.t.pl_off;
    const float2* __restrict__ P1 = P0 + p.t.pl_len;
    for (int f = tid; f <= N; f += NT) {
        const float2 a = __ldg(P0 + f), b = __ldg(P1 + f);
        A[f] = make_float2(a.x + b.x, a.y + b.y);
    }
    // overflow entries round by round: the targets of one round are distinct, a barrier orders the rounds
    for (int r = 0; r < p.t.ex_rounds; ++r) {
        __syncthreads();
        for (int i = tid; i < p.t.n_ex; i += NT) {
            const int4 q = __ldg(p.t.ex + i);
            if (q.w != 2 * r) continue;             // other rounds; folded entries: below
            float2 e = __ldg(Trow + q.y);
            if (q.z >= 0) { const float2 v = __ldg(Trow + q.z); e.x += v.x; e.y += v.y; }
            A[q.x].x += e.x; A[q.x].y += e.y;
        }
    }
    if (p.t.adjoint & 2) {
        __syncthreads();
        for (int f = 1 + tid; f <= p.t.pad_l; f += NT) {
            const float2 a = __ldg(P0 - f), b = __ldg(P1 - f);
            A[f].x += a.x + b.x; A[f].y -= a.y + b.y;
        }
        for (int f = 1 + tid; f <= p.t.pad_r; f += NT) {
            const float2 a = __ldg(P0 + N + f), b = __ldg(P1 + N + f);
            A[N - f].x += a.x + b.x; A[N - f].y -= a.y + b.y;
        }
        // overflow entries below DC / above Nyquist fold back conjugated, like the plane margins above: their targets
        // coincide with those of the margins and of the direct entries, so in a pass of their own (distinct targets
        // within a round)
        for (int r = 0; r < p.t.ex_rounds; ++r) {
            __syncthreads();
            for (int i = tid; i < p.t.n_ex; i += NT) {
                const int4 q = __ldg(p.t.ex + i);
                if (q.w != 2 * r + 1) continue;
                float2 e = __ldg(Trow + q.y);
                if (q.z >= 0) { const float2 v = __ldg(Trow + q.z); e.x += v.x; e.y += v.y; }
                A[q.x].x += e.x; A[q.x].y -= e.y;
            }
        }
    }
    __syncthreads();
    for (int kk = tid; kk <= N / 2; kk += NT) {
        const float2 rk = A[kk], rn = A[N - kk];
        if (kk == 0) {
            const float es = (p.t.adjoint & 2) ? 2.f : 1.f;
            const float a = rk.x * es, b = rn.x * es;
            A[0] = make_float2(a + b, a - b);
        } else {
            const float2 wk = __ldg(p.t.post_tw + kk);
            const float2 E = make_float2(rk.x + rn.x, rk.y - rn.y);
            const float2 O = make_float2(rk.x - rn.x, rk.y + rn.y);
            const float2 t = make_float2(fmaf(O.x, wk.x, O.y * wk.y), fmaf(O.y, wk.x, -O.x * wk.y));   // O conj(w)
            A[kk] = make_float2(E.x - t.y, E.y + t.x);
            A[N - kk] = make_float2(E.x + t.y, t.x - E.y);
        }
    }
    __syncthreads();
    const float2* Z = stockham<true>(A, B, N, p.t.n_fac, p.t.fac, p.t.wN, p.t.wP);
    const long long tb = (p.k0 + k - 1) * (long long)p.t.hop - p.t0;
    float* __restrict__ yr = p.x + row * p.x_row_stride;
    const bool accumulate = p.parity != 0;
    const bool second_store = !accumulate || (k + 1 >= p.S);
    const bool first_to_halo = (k == 0);
    float* __restrict__ halo = (p.halo_out != nullptr && p.k0 > 0) ? p.halo_out + (long long)row * p.t.hop : nullptr;
    const bool add1 = accumulate, add2 = accumulate && !second_store;
    const float2* __restrict__ tw2 = reinterpret_cast<const float2*>(p.t.tukey);
    for (int n = tid; n < N; n += NT) {
        float2 z = Z[n];
        if (p.t.adjoint & 2) { const float2 w = __ldg(tw2 + n); z.x *= w.x; z.y *= w.y; }
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

// ------------------------------------------------------------------------------------------
// The reference's second pass over the bins (nsigtf.py:63-80, k == 1) adds, for every bin 1 .. J-2, a "mirrored" copy
// at position L - pos_j built as conj(cat(t[1:], flip(t[1:]))) of the bin's coefficient spectrum t = FFT_M(c_j).  It
// matters only where that copy lands in the kept half [0, L/2], i.e. for a bin that reaches below DC (pos_j < M_j / 2):
// spectrum position f = m - pos_j (m in [pos_j, M_j/2)) receives conj(t[m + 1]) * gd_mirror[m] * M_j.  In the reference's
// rotated-slice bookkeeping this term picks up -/+ i on even / odd slices on top of the bin's sign (DESIGN.md): the entry
// weight carries (-1)^(pos/2) M gd / L, the kernel the slice parity.  One thread per (unit, position f): for every
// mirrored bin that reaches f, in bin order, t[m + 1] by a direct M-term sum over the caller's coefficients; then ONE
// read-modify-write of the plane-0 position (after bins_inv_kernel, before the slice kernel, same stream).  No two
// threads touch one position and the terms are added in a fixed order, so the result is deterministic.
__global__ void mirror_fix_kernel(const __grid_constant__ SlicqBinsParams p) {
    const int nf = p.t.mir_nf;
    const long long total = (long long)p.n_rs * nf;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int u = (int)(i / nf), f = (int)(i - (long long)u * nf);
        const int rs = p.rs0 + u;
        const int row = rs / p.S, k = rs - row * p.S;
        const int rowx = p.x_rows ? row % p.x_rows : row;
        const bool odd = ((p.k0 + k) & 1) != 0;
        float2* dst = p.spec + (long long)u * p.spec_stride + p.t.pl_off + f;
        float2 sum = *dst;
        for (int bi = 0; bi < p.t.n_mir_bins; ++bi) {
            const SlicqMirrorBin mb = p.t.mir_bins[bi];
            if (f >= mb.count) continue;
            const SlicqMirrorEntry me = p.t.mir[mb.first + f];
            const SlicqBucketArg& b = p.b[mb.bucket];
            const float2* c = b.ptr + rowx * b.s_row + mb.f_in_bucket * b.s_bin + k * b.s_slice;
            const float* mk = b.mptr ? b.mptr + row * b.ms_row + mb.f_in_bucket * b.ms_bin + k * b.ms_slice : nullptr;
            const float2* __restrict__ tw = p.t.tw + b.tw_off;           // exp(-2 pi i j / M)
            float2 acc = make_float2(0.f, 0.f);
            int idx = 0;
            for (int n = 0; n < b.M; ++n) {
                float2 v = c[n];
                if (mk) { v.x *= mk[n]; v.y *= mk[n]; }
                const float2 w = __ldg(tw + idx);
                acc.x += v.x * w.x - v.y * w.y;
                acc.y += v.x * w.y + v.y * w.x;
                idx += me.m_src; if (idx >= b.M) idx -= b.M;
            }
            // conj(t) * weight * (-i on even, +i on odd global slices)
            const float2 ct = make_float2(acc.x * me.weight, -acc.y * me.weight);
            const float2 val = odd ? make_float2(-ct.y, ct.x) : make_float2(ct.y, -ct.x);
            sum.x += val.x; sum.y += val.y;
        }
        *dst = sum;
    }
}

// Transpose of mirror_fix_kernel under <a, b> = Re(conj(a) b), for the analysis entry of a SLICQ_PLAN_ADJOINT_OF_SYNTHESIS
// plan.  The forward term adds s i w conj(sum_n c[n] e^{-2 pi i n q / M}) at position f (q = m_src, w the entry weight,
// s = -1 / +1 on even / odd global slices); its transpose is
//     c[n] += s i (L w) conj(H[f]) e^{+2 pi i n q / M},
// H the adjoint plan's padded half spectrum (2/L, 1/L at DC, folded in; L w undoes the 1/L the weight carries for the
// slice IFFT).  Runs after bins_fwd_kernel on the same stream.  One thread per (unit, mirrored bin, n) sums the bin's
// entries in order and updates c[n] once: no atomics, deterministic.  In the mask-gradient mode (p.mask_grad) the bins
// kernel has stored Re(conj(X) c) instead of c, X the mixture; the same term then goes to that gradient:
//     grad[n] += Re(conj(X[n]) v),  X read at mixture row row % x_rows.
__global__ void mirror_adj_kernel(const __grid_constant__ SlicqBinsParams p) {
    const int nc = p.t.mir_nc;
    const long long total = (long long)p.n_rs * nc;
    const float Lf = (float)p.t.L;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int u = (int)(i / nc);
        int n = (int)(i - (long long)u * nc), bi = 0;
        while (n >= p.b[p.t.mir_bins[bi].bucket].M) { n -= p.b[p.t.mir_bins[bi].bucket].M; ++bi; }
        const SlicqMirrorBin mb = p.t.mir_bins[bi];
        const SlicqBucketArg& b = p.b[mb.bucket];
        const int rs = p.rs0 + u;
        const int row = rs / p.S, k = rs - row * p.S;
        const float2* __restrict__ H = p.spec + (long long)u * p.spec_stride + p.t.pad_l;
        const float2* __restrict__ tw = p.t.tw + b.tw_off;           // exp(-2 pi i j / M)
        float2 acc = make_float2(0.f, 0.f);                          // sum_f (L w) conj(H[f] e^{-2 pi i n q / M})
        for (int f = 0; f < mb.count; ++f) {
            const SlicqMirrorEntry me = p.t.mir[mb.first + f];
            const float2 hw = cmul(H[f], __ldg(tw + (n * me.m_src) % b.M));
            const float a = Lf * me.weight;
            acc.x += a * hw.x; acc.y -= a * hw.y;
        }
        const bool odd = ((p.k0 + k) & 1) != 0;                       // times +i on odd, -i on even global slices
        const float2 v = odd ? make_float2(-acc.y, acc.x) : make_float2(acc.y, -acc.x);
        if (p.mask_grad) {
            const float2 x = b.ptr[(p.x_rows ? row % p.x_rows : row) * b.s_row + mb.f_in_bucket * b.s_bin + k * b.s_slice + n];
            float* gm = b.nptr + row * b.ms_row + mb.f_in_bucket * b.ms_bin + k * b.ms_slice + n;
            *gm += mask_grad_of(x, v);
            continue;
        }
        float2* c = b.ptr + row * b.s_row + mb.f_in_bucket * b.s_bin + k * b.s_slice + n;
        float2 cv = *c;
        cv.x += v.x; cv.y += v.y;
        *c = cv;
    }
}

// ------------------------------------------------------------------------------------------
// The long bin (SlicqLongBinParams: the Nyquist bin of a band-limited filterbank, too long for the bins kernels' register
// codelets).  The formulas of the bins kernels (k_bins.cu), for one transform of length M per CTA on the Stockham engine
// above, after bins_fwd_kernel / bins_inv_kernel on the same stream:
//     analysis   c[n] = (-1)^n IDFT_M(H[hoff + m'] wf'[m'])[n]  -> the caller's bucket, and |c| (slicq_forward_norm);
//                in the mask-gradient mode Re(conj(X) c) instead, X the mixture at row row % x_rows
//     synthesis  T[off + m'] = wi'[m'] DFT_M((-1)^n c[n] (x mask[n], c from mixture row row % x_rows))[m'],
//                off = ovoff for the leading ov coefficients, toff for the others; and the gap zero-fill of the bucket
// Launch bound 3: the transform needs few registers, and short long bins (a few hundred coefficients) run 3 CTAs per SM.
__global__ void __launch_bounds__(SLICQ_GEN_THREADS, 3) long_bin_fwd_kernel(const __grid_constant__ SlicqLongBinParams p) {
    SLICQ_DYN_SMEM(float2, A);
    const int M = p.M, NT = SLICQ_GEN_THREADS, tid = threadIdx.x;
    float2* B = A + M;
    const int u = blockIdx.x;
    const int rs = p.rs0 + u;
    const int row = rs / p.S, k = rs - row * p.S;
    const float2* __restrict__ H = p.spec + (long long)u * p.spec_stride + p.hoff;
    for (int m = tid; m < M; m += NT) {
        const float2 h = H[m];
        const float w = __ldg(p.w + m);
        A[m] = make_float2(h.x * w, h.y * w);
    }
    __syncthreads();
    const float2* Z = stockham<true>(A, B, M, p.n_fac, p.fac, p.wM, p.wP);
    const SlicqBucketArg& b = p.b;
    const int rowx = p.mask_grad ? row % p.x_rows : row;
    float2* __restrict__ c = b.ptr + rowx * b.s_row + k * b.s_slice;
    float* __restrict__ aux = b.nptr ? b.nptr + row * b.ms_row + k * b.ms_slice : nullptr;
    for (int n = tid; n < M; n += NT) {
        float2 v = Z[n];
        if (n & 1) v = make_float2(-v.x, -v.y);
        if (p.mask_grad) { aux[n] = mask_grad_of(c[n], v); continue; }
        c[n] = v;
        if (aux) aux[n] = sqrtf(fmaf(v.x, v.x, v.y * v.y));
    }
}

__global__ void __launch_bounds__(SLICQ_GEN_THREADS, 3) long_bin_inv_kernel(const __grid_constant__ SlicqLongBinParams p) {
    SLICQ_DYN_SMEM(float2, A);
    const int M = p.M, NT = SLICQ_GEN_THREADS, tid = threadIdx.x;
    float2* B = A + M;
    const int u = blockIdx.x;
    const int rs = p.rs0 + u;
    const int row = rs / p.S, k = rs - row * p.S;
    const SlicqBucketArg& b = p.b;
    const float2* __restrict__ c = b.ptr + (p.x_rows ? row % p.x_rows : row) * b.s_row + k * b.s_slice;
    const float* __restrict__ mk = b.mptr ? b.mptr + row * b.ms_row + k * b.ms_slice : nullptr;
    for (int n = tid; n < M; n += NT) {
        float2 v = c[n];
        if (mk) { const float m = mk[n]; v.x *= m; v.y *= m; }
        if (n & 1) v = make_float2(-v.x, -v.y);
        A[n] = v;
    }
    __syncthreads();
    const float2* Z = stockham<false>(A, B, M, p.n_fac, p.fac, p.wM, p.wP);
    float2* __restrict__ T = p.spec + (long long)u * p.spec_stride;
    for (int m = tid; m < M; m += NT) {
        const float2 z = Z[m];
        const float w = __ldg(p.w + m);
        T[(m < p.ov ? p.ovoff : p.toff) + m] = make_float2(z.x * w, z.y * w);
    }
    // positions of the T planes that no bin covers and that this bucket owns (see SlicqDeviceTables)
    for (int e = 0; e < p.gap_n; ++e) {
        const int2 g = __ldg(p.gaps + e);
        for (int i = tid; i < g.y; i += NT) T[g.x + i] = make_float2(0.f, 0.f);
    }
}

extern "C" int slicq_long_bin_smem_bytes(int M) {
    const long long b = 2LL * M * (long long)sizeof(float2);
    return (M > 0 && b <= 220 * 1024) ? (int)b : -1;
}

extern "C" int slicq_launch_long_bin(const SlicqLongBinParams* p, int inverse, cudaStream_t s) {
    if (p->n_rs <= 0) return 0;
    const int smem = slicq_long_bin_smem_bytes(p->M);
    if (smem < 0) return -2;
    if (inverse) {
        if (slicq_smem_opt_in<long_bin_inv_kernel>(smem)) return -3;
        SLICQ_LAUNCH(long_bin_inv_kernel, dim3(p->n_rs), dim3(SLICQ_GEN_THREADS), smem, s, *p);
    } else {
        if (slicq_smem_opt_in<long_bin_fwd_kernel>(smem)) return -3;
        SLICQ_LAUNCH(long_bin_fwd_kernel, dim3(p->n_rs), dim3(SLICQ_GEN_THREADS), smem, s, *p);
    }
    return (int)cudaGetLastError();
}

extern "C" int slicq_generic_smem_bytes(int L) {
    const long long b = 2LL * (L / 2 + 2) * (long long)sizeof(float2);
    return (L > 0 && L % 4 == 0 && b <= 220 * 1024) ? (int)b : -1;
}

extern "C" int slicq_launch_slice_fwd_generic(const SlicqSliceParams* p, cudaStream_t s) {
    if (p->n_rs <= 0) return 0;
    const int smem = slicq_generic_smem_bytes(p->t.L);
    if (smem < 0) return -2;
    if (slicq_smem_opt_in<slice_fft_fwd_generic_kernel>(smem)) return -3;
    SLICQ_LAUNCH(slice_fft_fwd_generic_kernel, dim3(p->n_rs), dim3(SLICQ_GEN_THREADS), smem, s, *p);
    return (int)cudaGetLastError();
}

extern "C" int slicq_launch_slice_inv_generic(const SlicqSliceParams* p, cudaStream_t s) {
    if (p->n_rs <= 0) return 0;
    const int smem = slicq_generic_smem_bytes(p->t.L);
    if (smem < 0) return -2;
    if (slicq_smem_opt_in<slice_fft_inv_generic_kernel>(smem)) return -3;
    SlicqSliceParams sp;
    const unsigned ctas = slicq_parity_ctas(*p, sp);
    if (!ctas) return 0;
    SLICQ_LAUNCH(slice_fft_inv_generic_kernel, dim3(ctas), dim3(SLICQ_GEN_THREADS), smem, s, sp);
    return (int)cudaGetLastError();
}

extern "C" int slicq_launch_mirror_fix(const SlicqBinsParams* p, cudaStream_t s) {
    if (p->t.n_mir <= 0 || p->n_rs <= 0) return 0;
    const long long total = (long long)p->n_rs * p->t.mir_nf;
    const int blocks = (int)((total + 127) / 128 > 4096 ? 4096 : (total + 127) / 128);
    SLICQ_LAUNCH(mirror_fix_kernel, dim3(blocks), dim3(128), 0, s, *p);
    return (int)cudaGetLastError();
}

extern "C" int slicq_launch_mirror_adj(const SlicqBinsParams* p, cudaStream_t s) {
    if (p->t.n_mir <= 0 || p->n_rs <= 0) return 0;
    const long long total = (long long)p->n_rs * p->t.mir_nc;
    const int blocks = (int)((total + 127) / 128 > 4096 ? 4096 : (total + 127) / 128);
    SLICQ_LAUNCH(mirror_adj_kernel, dim3(blocks), dim3(128), 0, s, *p);
    return (int)cudaGetLastError();
}
