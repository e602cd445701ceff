// Batched small-FFT engine of the analysis (per-bin IFFT) and synthesis (per-bin FFT) kernels.
//
// A CTA ("job") owns ONE bucket (F bins of equal length M) and a contiguous range of (row,slice)
// units, and walks the range `gt` units at a time.  Everything that does not depend on the unit
// -- the thread's bin, its position inside the transform, its window coefficients -- is computed
// once per job and kept in registers; the per-unit work is loads, one register codelet, a
// shared-memory transpose, the second codelet and stores.  Because a CTA executes a single M for
// its whole life, only that size's straight-line codelets are live in the instruction cache.
//
// Index conventions.  Windows and spectrum reads use the *centred* order m' = m~ + M/2 with
// m~ in [-M/2, M/2) the offset from the bin centre: x'[m'] = H[pos - M/2 + m'] (contiguous, no
// wrap, no reflection thanks to the mirrored margins of H).  The reference's ifftshift is the
// circular shift by M/2, which in the transform domain is the sign (-1)^n:
//     analysis   c[n]  = (-1)^n * IDFT_M(x' * wf')[n]
//     synthesis  T'[m'] = wi'[m'] * DFT_M((-1)^n c[n])[m']
// Plans per M (fft_sizes.inc): kind 1 = one thread per transform, kind 2 = A x B Cooley-Tukey
// through shared memory, kind 3 = prime P >= 29 times R via the real symmetric half transforms.
#pragma once
#include "slicq_common.cuh"
#include "dft_codelets.cuh"

// independent 16-byte loads in flight per thread in the input loop of the single-thread synthesis transforms
constexpr int kSynSingleLoads = 4;
// two-pass synthesis transforms with A + B up to this bound prefetch their next inputs into registers (see syn_two_pass)
constexpr int kSynPipeMax = 26;

struct JobCtx {
    int u0, u1;     // unit range of this job (indices local to the chunk)
    int F;          // bins in the bucket
    int gt;         // units per iteration
    int first_bin;
    int rs0, S;     // chunk origin and slices per row: unit g is (row, k) = divmod(rs0 + g, S)
    int x_rows;     // masked synthesis: mixture rows (0 = plain)
    bool aux;       // a second tensor (synthesis: mask, analysis: magnitude or mask-gradient output) is addressed through ms_*
};

SLICQ_DEVFN float2 cneg_if(float2 v, bool neg) { return neg ? make_float2(-v.x, -v.y) : v; }

// The first SLOT_BYTES of a job's shared memory hold, for the units of the current iteration, the
// element offset of (row, bin f, slice k, 0) in the caller's bucket tensor: slot = gs * F + f.
// One integer division per slot and iteration instead of one per coefficient.
// In masked synthesis (mixture * mask fused into the load, reference: phase.py:96-113 /
// model.py:258-265) a second table [256, 512) holds the offsets into the mask tensor.  In the mask-gradient analysis
// the first table addresses the mixture (row % x_rows) and the second the gradient (output row).
#define SLICQ_SLOT_BYTES 4096
SLICQ_DEVFN void fill_slot_off(long long* so, const SlicqBucketArg& b, const JobCtx& j, int base, int ng, int x_rows) {
    for (int t = threadIdx.x; t < ng * j.F; t += blockDim.x) {
        const int gs = t / j.F, f = t - gs * j.F;
        const int rs = j.rs0 + base + gs;
        const int row = rs / j.S, k = rs - row * j.S;
        const int rowx = x_rows ? row % x_rows : row;
        so[t] = rowx * b.s_row + f * b.s_bin + k * b.s_slice;
        if (j.aux) so[256 + t] = row * b.ms_row + f * b.ms_bin + k * b.ms_slice;
    }
}
SLICQ_DEVFN float2 cscale(float2 v, float s) { return make_float2(v.x * s, v.y * s); }
SLICQ_DEVFN float cmag(float2 v) { return sqrtf(fmaf(v.x, v.x, v.y * v.y)); }

// =========================================================================================
// kind 1
// =========================================================================================
// Analysis transforms: MG = mask-gradient epilogue (SlicqBinsParams::mask_grad, slicq_forward_mask_grad).  A compile-time
// mode with a kernel of its own (bins_fwd_mask_grad_kernel): bins_fwd_kernel keeps the code and registers of the plain
// analysis (a run-time branch in the stores cost 0.7 % of the default bench step on a B200 at 1000 W).
template <int M, bool MG>
SLICQ_DEVFN void ana_single(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, float2* sm) {
    constexpr int PITCH = M + 1;
    const int tid = threadIdx.x;
    const int gs = tid / j.F, f = tid - gs * j.F;
    const bool act = gs < j.gt;
    // window of the thread's bin: registers for the short transforms, shared memory (behind the
    // stage) for M > 24, where the codelet needs the registers itself
    constexpr bool WREG = M <= 24;
    float w[WREG ? M : 1];
    int hoff = 0;
    if (act) {
        const int bin = j.first_bin + f;
        const int coff = __ldg(p.t.bin_coff + bin);
        hoff = p.t.pad_l + __ldg(p.t.bin_pos + bin) - M / 2;
        if (WREG) {
#pragma unroll
            for (int m = 0; m < (WREG ? M : 1); ++m) w[m] = __ldg(p.t.wf + coff + m);
        }
    }
    long long* so = reinterpret_cast<long long*>(sm);
    sm += SLICQ_SLOT_BYTES / sizeof(float2);
    float2* stage = sm + (gs * j.F + f) * PITCH;
    const float* wsm = reinterpret_cast<const float*>(sm + j.gt * j.F * PITCH) + f * M;
    if (!WREG) {
        float* wd = reinterpret_cast<float*>(sm + j.gt * j.F * PITCH);
        const int coff0 = __ldg(p.t.bin_coff + j.first_bin);
        for (int t = tid; t < j.F * M; t += blockDim.x) wd[t] = __ldg(p.t.wf + coff0 + t);
        __syncthreads();
    }
    for (int base = j.u0; base < j.u1; base += j.gt) {
        const int g = base + gs;
        const int ng = (j.u1 - base < j.gt) ? (j.u1 - base) : j.gt;
        fill_slot_off(so, b, j, base, ng, MG ? p.x_rows : 0);
        if (act && g < j.u1) {
            const float4* h = reinterpret_cast<const float4*>(p.spec + (long long)g * p.spec_stride + hoff);
            float2 v[M];
#pragma unroll
            for (int m = 0; m < M; m += 2) {
                const float4 x = h[m >> 1];
                const float w0 = WREG ? w[WREG ? m : 0] : wsm[m], w1 = WREG ? w[WREG ? m + 1 : 0] : wsm[m + 1];
                v[m] = make_float2(x.x * w0, x.y * w0);
                v[m + 1] = make_float2(x.z * w1, x.w * w1);
            }
            dft<M, true>(v);
#pragma unroll
            for (int n = 0; n < M; ++n) stage[n] = cneg_if(v[n], n & 1);
        }
        __syncthreads();
        for (int t = tid; t < ng * j.F * M; t += blockDim.x) {
            const int slot = t / M, n = t - slot * M;
            const float2 c = sm[slot * PITCH + n];
            if (MG) {
                b.nptr[so[256 + slot] + n] = mask_grad_of(b.ptr[so[slot] + n], c);
                continue;
            }
            b.ptr[so[slot] + n] = c;
            if (b.nptr != nullptr) b.nptr[so[256 + slot] + n] = cmag(c);
        }
        __syncthreads();
    }
}

// synthesis: coefficients come in through shared memory (coalesced 16-byte loads), every thread
// transforms one row in place, and the windowed spectra of a unit -- one contiguous block
// [coff_first, coff_first + F*M) of the packed row T -- leave through shared memory again.
template <int M>
SLICQ_DEVFN void syn_single(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, float2* sm) {
    constexpr int PITCH = M + 1;
    const int tid = threadIdx.x;
    const int gs = tid / j.F, f = tid - gs * j.F;
    const bool act = gs < j.gt;
    const int coff0 = __ldg(p.t.bin_coff + j.first_bin);
    const int FM = j.F * M;
    long long* so = reinterpret_cast<long long*>(sm);
    sm += SLICQ_SLOT_BYTES / sizeof(float2);
    float2* stage = sm + (gs * j.F + f) * PITCH;
    // the bucket's dual windows (contiguous in wi) and the T-row offsets of its bins live behind the stage; both
    // are applied on the way out: no per-thread window registers next to the M-point codelet
    float* wsm = reinterpret_cast<float*>(sm + j.gt * j.F * PITCH);
    int* tob = reinterpret_cast<int*>(wsm + FM);           // [F] {offset of m' = 0, overflow count, overflow offset}
    for (int t = tid; t < FM; t += blockDim.x) wsm[t] = __ldg(p.t.wi + coff0 + t);
    for (int t = tid; t < j.F; t += blockDim.x) {
        tob[3 * t] = __ldg(p.t.bin_toff + j.first_bin + t);
        tob[3 * t + 1] = __ldg(p.t.bin_ov + j.first_bin + t);
        tob[3 * t + 2] = __ldg(p.t.bin_ovoff + j.first_bin + t);
    }
    const bool vec = b.mptr == nullptr && ((reinterpret_cast<uintptr_t>(b.ptr) & 15) == 0) &&
                     (((b.s_row | b.s_bin | b.s_slice) & 1) == 0);
    for (int base = j.u0; base < j.u1; base += j.gt) {
        const int ng = (j.u1 - base < j.gt) ? (j.u1 - base) : j.gt;
        fill_slot_off(so, b, j, base, ng, j.x_rows);
        __syncthreads();
        if (vec) {
            // four independent 16-byte loads in flight per thread (a rolled loop would wait for each in turn)
            constexpr int U = kSynSingleLoads;
            const int tot = ng * j.F * (M / 2);
            for (int t0 = tid; t0 < tot; t0 += U * blockDim.x) {
                float4 v[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int t = t0 + u * blockDim.x;
                    if (t < tot) {
                        const int slot = t / (M / 2), n = 2 * (t - slot * (M / 2));
                        v[u] = *reinterpret_cast<const float4*>(b.ptr + so[slot] + n);
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int t = t0 + u * blockDim.x;
                    if (t < tot) {
                        const int slot = t / (M / 2), n = 2 * (t - slot * (M / 2));
                        sm[slot * PITCH + n] = make_float2(v[u].x, v[u].y);
                        sm[slot * PITCH + n + 1] = make_float2(v[u].z, v[u].w);
                    }
                }
            }
        } else if (b.mptr == nullptr) {
            for (int t = tid; t < ng * j.F * M; t += blockDim.x) {
                const int slot = t / M, n = t - slot * M;
                sm[slot * PITCH + n] = b.ptr[so[slot] + n];
            }
        } else {
            for (int t = tid; t < ng * j.F * M; t += blockDim.x) {
                const int slot = t / M, n = t - slot * M;
                sm[slot * PITCH + n] = cscale(b.ptr[so[slot] + n], b.mptr[so[256 + slot] + n]);
            }
        }
        __syncthreads();
        if (act && base + gs < j.u1) {
            float2 v[M];
#pragma unroll
            for (int n = 0; n < M; ++n) v[n] = cneg_if(stage[n], n & 1);
            dft<M, false>(v);
#pragma unroll
            for (int m = 0; m < M; ++m) stage[m] = v[m];
        }
        __syncthreads();
        // rows of T are 16-byte aligned, bin offsets / overflow counts are even: two coefficients per store
        for (int t = tid; t < ng * (FM / 2); t += blockDim.x) {
            const int g = t / (FM / 2), e = 2 * (t - g * (FM / 2));
            const int fb = e / M, n = e - fb * M;
            const float2* src = sm + (g * j.F + fb) * PITCH + n;
            const float w0 = wsm[e], w1 = wsm[e + 1];
            const int off = (n < tob[3 * fb + 1] ? tob[3 * fb + 2] : tob[3 * fb]) + n;
            *reinterpret_cast<float4*>(p.spec + (long long)(base + g) * p.spec_stride + off) =
                make_float4(src[0].x * w0, src[0].y * w0, src[1].x * w1, src[1].y * w1);
        }
    }
}

// =========================================================================================
// kind 2 : M = A * B, A >= B
// =========================================================================================
// analysis: x'[B*n1 + n2] -> X[k1 + A*k2];  pass 1 = DFT-A (hoisted window), pass 2 = DFT-B (runs of A to HBM)
template <int M, int A, int B, bool MG>
SLICQ_DEVFN void ana_two_pass(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, float2* sm) {
    static_assert(A * B == M, "bad split");
    constexpr int BP = (B % 2 == 0) ? B + 1 : B;
    constexpr int PER = A * BP;
    const int tid = threadIdx.x;
    const int per1 = j.F * B;
    const int gs1 = tid / per1, r1 = tid - gs1 * per1;
    const int f1 = r1 / B, n2 = r1 - f1 * B;
    const bool act1 = gs1 < j.gt;
    float w[A];
    int hoff = 0;
    if (act1) {
        const int bin = j.first_bin + f1;
        const int coff = __ldg(p.t.bin_coff + bin);
        hoff = p.t.pad_l + __ldg(p.t.bin_pos + bin) - M / 2 + n2;
#pragma unroll
        for (int n1 = 0; n1 < A; ++n1) w[n1] = __ldg(p.t.wf + coff + B * n1 + n2);
    }
    long long* so = reinterpret_cast<long long*>(sm);
    sm += SLICQ_SLOT_BYTES / sizeof(float2);
    float2* y1 = sm + (gs1 * j.F + f1) * PER + n2;
    // the job's twiddles, transposed to [k1][n2], in shared memory behind the stage (immediate offsets in pass 1)
    float2* twsm = sm + j.gt * j.F * PER;
    {
        const float2* __restrict__ tw = p.t.tw + b.tw_off;
        for (int t = tid; t < M; t += blockDim.x) { const int k1 = t / B, c2 = t - k1 * B; twsm[t] = __ldg(tw + c2 * k1); }
    }
    const float2* twp = twsm + n2;
    __syncthreads();
    for (int base = j.u0; base < j.u1; base += j.gt) {
        const int g = base + gs1;
        const int ng = (j.u1 - base < j.gt) ? (j.u1 - base) : j.gt;
        fill_slot_off(so, b, j, base, ng, MG ? p.x_rows : 0);
        if (act1 && g < j.u1) {
            const float2* h = p.spec + (long long)g * p.spec_stride + hoff;
            float2 v[A];
#pragma unroll
            for (int n1 = 0; n1 < A; ++n1) {
                const float2 x = h[B * n1];
                v[n1] = make_float2(x.x * w[n1], x.y * w[n1]);
            }
            dft<A, true>(v);
            y1[0] = v[0];
#pragma unroll
            for (int k1 = 1; k1 < A; ++k1)
                y1[k1 * BP] = cneg_if(cmul_conj(v[k1], twp[k1 * B]), k1 & 1);  // (-1)^k1 folded here
        }
        __syncthreads();
        for (int t = tid; t < ng * j.F * A; t += blockDim.x) {
            const int slot = t / A, k1 = t - slot * A;
            const float2* src = sm + slot * PER + k1 * BP;
            float2 v[B];
#pragma unroll
            for (int n = 0; n < B; ++n) v[n] = src[n];
            dft<B, true>(v);
            float2* o = b.ptr + so[slot] + k1;
            if (MG) {
                float* og = b.nptr + so[256 + slot] + k1;
#pragma unroll
                for (int k2 = 0; k2 < B; ++k2) og[A * k2] = mask_grad_of(o[A * k2], cneg_if(v[k2], (A * k2) & 1));
                continue;
            }
#pragma unroll
            for (int k2 = 0; k2 < B; ++k2) o[A * k2] = cneg_if(v[k2], (A * k2) & 1);
            if (b.nptr != nullptr) {
                float* on = b.nptr + so[256 + slot] + k1;
#pragma unroll
                for (int k2 = 0; k2 < B; ++k2) on[A * k2] = cmag(v[k2]);
            }
        }
        __syncthreads();
    }
}

// synthesis: x[B*n1 + n2] -> X[k1 + A*k2];  same shape as the analysis: pass 1 = DFT-A with the
// thread's (unit, bin, n2) fixed for the whole job (runs of B from the caller's tensor), pass 2 =
// DFT-B, dual window, runs of A into the packed row T.
// OVR: a bin may divert more than its first run of outputs to its overflow slot (bins_inv_ovr_kernel, plans whose bins
// crowd together near DC); a compile-time mode, so that bins_inv_kernel keeps its one select on the first run.
template <int M, int A, int B, bool OVR>
SLICQ_DEVFN void syn_two_pass(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, float2* sm) {
    static_assert(A * B == M, "bad split");
    constexpr int BP = (B % 2 == 0) ? B + 1 : B;
    constexpr int PER = A * BP;
    const int tid = threadIdx.x;
    const int per1 = j.F * B;
    const int gs1 = tid / per1, r1 = tid - gs1 * per1;
    const int f1 = r1 / B, n2 = r1 - f1 * B;
    const bool act1 = gs1 < j.gt;
    const bool odd = n2 & 1;
    // per-slot constants of pass 2 (do not change over the job): unit offset gs | bin << 16, T-row offset of the bin,
    // its overflow count and overflow offset (leading outputs of a bin that overlaps its plane neighbour)
    int4* sc = reinterpret_cast<int4*>(sm);
    sm += SLICQ_SLOT_BYTES / sizeof(float2);
    for (int t = tid; t < j.gt * j.F; t += blockDim.x) {
        const int gs = t / j.F, f = t - gs * j.F;
        sc[t] = make_int4(gs | (f << 16), __ldg(p.t.bin_toff + j.first_bin + f), __ldg(p.t.bin_ov + j.first_bin + f),
                          __ldg(p.t.bin_ovoff + j.first_bin + f));
    }
    float2* y1 = sm + (gs1 * j.F + f1) * PER + n2;
    // The job's twiddles, transposed to [k1][n2], and the bucket's dual windows live in shared memory
    // behind the stage: pass 1 / pass 2 read them at immediate offsets instead of computing global
    // addresses and waiting for L1 / L2 between the codelet and the stores.
    float2* twsm = sm + j.gt * j.F * PER;
    float* wsm = reinterpret_cast<float*>(twsm + M);
    const int coff_first = __ldg(p.t.bin_coff + j.first_bin);
    {
        const float2* __restrict__ tw = p.t.tw + b.tw_off;
        for (int t = tid; t < M; t += blockDim.x) { const int k1 = t / B, c2 = t - k1 * B; twsm[t] = __ldg(tw + c2 * k1); }
        for (int t = tid; t < j.F * M; t += blockDim.x) wsm[t] = __ldg(p.t.wi + coff_first + t);
    }
    const float2* twp = twsm + n2;
    __syncthreads();
    // Software pipeline (sizes whose two register sets fit, A + B <= kSynPipeMax): the inputs of the NEXT group of units are
    // requested right after pass 1 has put its outputs into shared memory, so that they travel during the barrier and pass 2.
    constexpr bool PIPE = (A + B <= kSynPipeMax);
    float2 v[A];
    int rowk[2] = {0, 0};           // (row, slice) of the unit whose inputs sit in v
    auto request = [&](int base) {
        const int g = base + gs1;
        if (act1 && g < j.u1) {
            const int rs = j.rs0 + g;
            const int row = rs / j.S, k = rs - row * j.S;
            const int rowx = j.x_rows ? row % j.x_rows : row;
            const float2* src = b.ptr + rowx * b.s_row + f1 * b.s_bin + k * b.s_slice + n2;
#pragma unroll
            for (int n1 = 0; n1 < A; ++n1) v[n1] = src[B * n1];
            rowk[0] = row; rowk[1] = k;
        }
    };
    if (PIPE) request(j.u0);
    for (int base = j.u0; base < j.u1; base += j.gt) {
        const int g = base + gs1;
        if (!PIPE) request(base);
        if (act1 && g < j.u1) {
#pragma unroll
            for (int n1 = 0; n1 < A; ++n1) v[n1] = cneg_if(v[n1], odd != (((B * n1) & 1) != 0));  // (-1)^(B n1 + n2)
            if (b.mptr != nullptr) {
                const float* msrc = b.mptr + rowk[0] * b.ms_row + f1 * b.ms_bin + rowk[1] * b.ms_slice + n2;
#pragma unroll
                for (int n1 = 0; n1 < A; ++n1) v[n1] = cscale(v[n1], msrc[B * n1]);
            }
            dft<A, false>(v);
            y1[0] = v[0];
#pragma unroll
            for (int k1 = 1; k1 < A; ++k1) y1[k1 * BP] = cmul(v[k1], twp[k1 * B]);
        }
        if (PIPE && base + j.gt < j.u1) request(base + j.gt);
        __syncthreads();
        const int ng = (j.u1 - base < j.gt) ? (j.u1 - base) : j.gt;
        for (int t = tid; t < ng * j.F * A; t += blockDim.x) {
            const int slot = t / A, k1 = t - slot * A;
            const int4 c = sc[slot];
            const float2* src = sm + slot * PER + k1 * BP;
            float2 v[B];
#pragma unroll
            for (int n = 0; n < B; ++n) v[n] = src[n];
            dft<B, false>(v);
            float2* row = p.spec + (long long)(base + (c.x & 0xffff)) * p.spec_stride;
            float2* o = row + c.y + k1;
            const float* wp = wsm + (c.x >> 16) * M + k1;
            if (OVR) {   // any output k1 + A k2 below the overflow count goes to the overflow slot
#pragma unroll
                for (int k2 = 0; k2 < B; ++k2) {
                    const float w = wp[A * k2];
                    float2* ok = (k1 + A * k2 < c.z) ? row + c.w + k1 + A * k2 : o + A * k2;
                    *ok = make_float2(v[k2].x * w, v[k2].y * w);
                }
                continue;
            }
            // without OVR overflow counts never exceed A (slicq_plan_create): only output k2 = 0 can be diverted
            {
                const float w = wp[0];
                float2* o0 = (k1 < c.z) ? row + c.w + k1 : o;
                *o0 = make_float2(v[0].x * w, v[0].y * w);
            }
#pragma unroll
            for (int k2 = 1; k2 < B; ++k2) {
                const float w = wp[A * k2];
                o[A * k2] = make_float2(v[k2].x * w, v[k2].y * w);
            }
        }
        __syncthreads();
    }
}

// =========================================================================================
// kind 3 : M = P * R, P prime >= 29, R in {4, 8}
// =========================================================================================
// The DFT-P is the streamed symmetric direct form split BY OUTPUTS over NP threads (Dftp<P, NP>, gen_codelets.py):
// packed complex FFMA2 with immediate twiddles, the accumulators the only long-lived registers.  The centring sign
// (-1)^n splits over the two index parts: a compile-time rotation by R/2 of the DFT-R side and a sign folded into the
// job's twiddle table.
template <int M> struct PrimeSrcSyn {      // synthesis pass 2: column n2 = 0 .. P-1, contiguous in shared memory
    const float2* p;
    SLICQ_DEVFN cpx ld(int n) const { return cpx_ld(p + n); }
};
struct PrimeSrcAna {                       // analysis pass 1: x'[R n + n2] * window, straight from the padded spectrum
    const float2* p; const float* w; int R;
    SLICQ_DEVFN cpx ld(int n) const { return cmulr(cpx_ld(p + R * n), w[R * n]); }
};
struct PrimeDstSyn {                       // synthesis pass 2: output k2 -> T[base + R k2] * window
    float2* o; const float* w; int R; int ovd;    // ovd: offset of the overflow slot relative to the plane slot, 0 = none
    SLICQ_DEVFN void st(int k, cpx v) const { cpx_st(o + R * k + (k == 0 ? ovd : 0), cmulr(v, w[R * k])); }
};
struct PrimeDstSynOvr {                    // the same when the overflow may span several runs (syn_prime OVR)
    float2* o; const float* w; int R; int ovd; int kov;    // outputs k < kov go to the overflow slot
    SLICQ_DEVFN void st(int k, cpx v) const { cpx_st(o + R * k + (k < kov ? ovd : 0), cmulr(v, w[R * k])); }
};
struct PrimeDstAna {                       // analysis pass 1: output k1 -> stage[k1 * RP + n2] * twiddle
    float2* o; const float2* tw; int RP, R;
    SLICQ_DEVFN void st(int k, cpx v) const { cpx_st(o + RP * k, k == 0 ? v : cmulw(v, tw[R * k])); }
};
constexpr __host__ __device__ int prime_parts(int P) { return P <= 41 ? 2 : (P <= 61 ? 3 : 4); }   // gen_codelets.py PRIME_PARTS

// analysis (prime first): x'[R*n1 + n2], n1 in [0,P) -> X[k1 + P*k2]
template <int M, int P, int R, bool MG>
SLICQ_DEVFN void ana_prime(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, float* smf) {
    static_assert(P * R == M && R % 2 == 0, "bad split");
    constexpr int NP = (P <= 41 ? 2 : (P <= 61 ? 3 : 4)), RP = R + 1, PER = P * RP;
    typedef Dftp<P, NP, true> D;
    const int tid = threadIdx.x;
    long long* so = reinterpret_cast<long long*>(smf);
    float2* sm = reinterpret_cast<float2*>(smf + SLICQ_SLOT_BYTES / sizeof(float));
    // job twiddles [k1][n2] = conj(exp(-2 pi i n2 k1 / M)) (-1)^k1, the bucket's analysis windows and the spectrum offset of
    // each bin in shared memory behind the stage
    float2* twsm = sm + (size_t)j.gt * j.F * PER;
    float* wsm = reinterpret_cast<float*>(twsm + M);
    int* hoff = reinterpret_cast<int*>(wsm + j.F * M);
    {
        const float2* __restrict__ tw = p.t.tw + b.tw_off;
        const int coff_first = __ldg(p.t.bin_coff + j.first_bin);
        for (int t = tid; t < M; t += blockDim.x) {
            const int k1 = t / R, c2 = t - k1 * R;
            float2 w = __ldg(tw + c2 * k1);
            w.y = -w.y;
            if (k1 & 1) { w.x = -w.x; w.y = -w.y; }
            twsm[t] = w;
        }
        for (int t = tid; t < j.F * M; t += blockDim.x) wsm[t] = __ldg(p.t.wf + coff_first + t);
        for (int t = tid; t < j.F; t += blockDim.x) hoff[t] = p.t.pad_l + __ldg(p.t.bin_pos + j.first_bin + t) - M / 2;
    }
    __syncthreads();
    for (int base = j.u0; base < j.u1; base += j.gt) {
        const int ng = (j.u1 - base < j.gt) ? (j.u1 - base) : j.gt;
        fill_slot_off(so, b, j, base, ng, MG ? p.x_rows : 0);
        // pass 1: DFT-P, task = (part, slot, n2 < R); a part's tasks fill whole warps
        const int ncol = ng * j.F * R, colp = (ncol + 31) & ~31;
        for (int t = tid; t < NP * colp; t += blockDim.x) {
            const int part = t / colp, c = t - part * colp;
            if (c >= ncol) continue;
            const int s = c / R, c2 = c - s * R;
            const int gs = s / j.F, f = s - gs * j.F;
            PrimeSrcAna src;
            src.p = p.spec + (long long)(base + gs) * p.spec_stride + hoff[f] + c2;
            src.w = wsm + f * M + c2; src.R = R;
            cpx o[D::NOUT];
            D::run(part, src, o);
            PrimeDstAna dst; dst.o = sm + s * PER + c2; dst.tw = twsm + c2; dst.RP = RP; dst.R = R;
            D::store(part, dst, o);
        }
        __syncthreads();
        // pass 2: DFT-R with its inputs rotated by R/2 ((-1)^k2 on the outputs, P odd), runs of P to the caller's tensor
        for (int t = tid; t < ng * j.F * P; t += blockDim.x) {
            const int s = t / P, k1 = t - s * P;
            const float2* src = sm + s * PER + k1 * RP;
            cpx v[R];
#pragma unroll
            for (int n = 0; n < R; ++n) v[n] = cpx_ld(src + (n + R / 2) % R);
            dft<R, true>(v);
            float2* o = b.ptr + so[s] + k1;
            if (MG) {
                float* og = b.nptr + so[256 + s] + k1;
#pragma unroll
                for (int k2 = 0; k2 < R; ++k2) og[P * k2] = mask_grad_of(o[P * k2], cpx_to(v[k2]));
                continue;
            }
#pragma unroll
            for (int k2 = 0; k2 < R; ++k2) cpx_st(o + P * k2, v[k2]);
            if (b.nptr != nullptr) {
                float* on = b.nptr + so[256 + s] + k1;
#pragma unroll
                for (int k2 = 0; k2 < R; ++k2) on[P * k2] = cmag(cpx_to(v[k2]));
            }
        }
        __syncthreads();
    }
}

// synthesis (prime last): x[P*n1 + n2], n1 in [0,R) -> X[k1 + R*k2], k2 in [0,P); OVR as in syn_two_pass
template <int M, int P, int R, bool OVR>
SLICQ_DEVFN void syn_prime(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, float* smf) {
    static_assert(P * R == M && R % 2 == 0, "bad split");
    constexpr int NP = (P <= 41 ? 2 : (P <= 61 ? 3 : 4));
    typedef Dftp<P, NP, false> D;
    const int tid = threadIdx.x;
    long long* so = reinterpret_cast<long long*>(smf);
    float2* sm = reinterpret_cast<float2*>(smf + SLICQ_SLOT_BYTES / sizeof(float));
    // job twiddles [k1][n2] = exp(-2 pi i n2 k1 / M) (-1)^n2, the bucket's dual windows and the T-row offsets of its bins
    // slot pitch M: pass 2 then reads column k1 of slot s at (s R + k1) P + n -- a single odd stride across the lanes
    // (a pitch of M + P put every half warp on 8 bank pairs: 2-way conflicts on the NP-times repeated loads of pass 2)
    float2* twsm = sm + (size_t)j.gt * j.F * (M + P);
    float* wsm = reinterpret_cast<float*>(twsm + M);
    const int coff_first = __ldg(p.t.bin_coff + j.first_bin);
    const int FM = j.F * M;
    int* tob = reinterpret_cast<int*>(wsm + FM);           // [F] {offset of m' = 0 in the T row, overflow count, overflow offset}
    {
        const float2* __restrict__ tw = p.t.tw + b.tw_off;
        for (int t = tid; t < M; t += blockDim.x) {
            const int k1 = t / P, c2 = t - k1 * P;
            float2 w = __ldg(tw + c2 * k1);
            if (c2 & 1) { w.x = -w.x; w.y = -w.y; }
            twsm[t] = w;
        }
        for (int t = tid; t < FM; t += blockDim.x) wsm[t] = __ldg(p.t.wi + coff_first + t);
        for (int t = tid; t < j.F; t += blockDim.x) {
            tob[3 * t] = __ldg(p.t.bin_toff + j.first_bin + t);
            tob[3 * t + 1] = __ldg(p.t.bin_ov + j.first_bin + t);
            tob[3 * t + 2] = __ldg(p.t.bin_ovoff + j.first_bin + t);
        }
    }
    for (int base = j.u0; base < j.u1; base += j.gt) {
        const int ng = (j.u1 - base < j.gt) ? (j.u1 - base) : j.gt;
        fill_slot_off(so, b, j, base, ng, j.x_rows);
        __syncthreads();
        // pass 1: DFT-R, task = (slot, n2 < P), input runs of P from the caller's tensor; (-1)^n1 = outputs rotated by R/2
        for (int t = tid; t < ng * j.F * P; t += blockDim.x) {
            const int s = t / P, c2 = t - s * P;
            const float2* src = b.ptr + so[s] + c2;
            cpx v[R];
#pragma unroll
            for (int n1 = 0; n1 < R; ++n1) v[n1] = cpx_ld(src + P * n1);
            if (b.mptr != nullptr) {
                const float* msrc = b.mptr + so[256 + s] + c2;
#pragma unroll
                for (int n1 = 0; n1 < R; ++n1) v[n1] = cmulr(v[n1], msrc[P * n1]);
            }
            dft<R, false>(v);
            float2* o = sm + s * M + c2;
            const float2* twp = twsm + c2;
#pragma unroll
            for (int k1 = 0; k1 < R; ++k1) cpx_st(o + k1 * P, cmulw(v[(k1 + R / 2) % R], twp[k1 * P]));
        }
        __syncthreads();
        // pass 2: DFT-P, task = (part, slot, k1); dual window, runs of R outputs to the plane row
        const int ncol = ng * j.F * R, colp = (ncol + 31) & ~31;
        for (int t = tid; t < NP * colp; t += blockDim.x) {
            const int part = t / colp, c = t - part * colp;
            if (c >= ncol) continue;
            const int s = c / R, k1 = c - s * R;
            const int gs = s / j.F, f = s - gs * j.F;
            PrimeSrcSyn<M> src; src.p = sm + s * M + k1 * P;
            cpx o[D::NOUT];
            D::run(part, src, o);
            if (OVR) {   // outputs k1 + R k2 below the overflow count: k2 < ceil((count - k1) / R)
                PrimeDstSynOvr dst;
                dst.o = p.spec + (long long)(base + gs) * p.spec_stride + tob[3 * f] + k1;
                dst.w = wsm + f * M + k1; dst.R = R;
                dst.ovd = tob[3 * f + 2] - tob[3 * f];
                dst.kov = (tob[3 * f + 1] - k1 + R - 1) / R;
                D::store(part, dst, o);
                continue;
            }
            PrimeDstSyn dst;
            dst.o = p.spec + (long long)(base + gs) * p.spec_stride + tob[3 * f] + k1;
            dst.w = wsm + f * M + k1; dst.R = R;
            dst.ovd = (k1 < tob[3 * f + 1]) ? tob[3 * f + 2] - tob[3 * f] : 0;
            D::store(part, dst, o);
        }
        __syncthreads();
    }
}
