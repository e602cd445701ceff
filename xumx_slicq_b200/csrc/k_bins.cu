// Stage 2 (analysis) and stage 3a (synthesis) of the sliCQT path: the ragged per-bin transforms.
//
//  bins_fwd_kernel  (reference: nsgt/nsgtf.py:50-81 + nsgt/slicq.py:13-33 `arrange`)
//      c_j[k, :] = (-1)^n IDFT_M( H_k[pos_j - M/2 + m'] * wf'_j[m'] ),  wf_j = g_j (-1)^(pos_j/2) / M_j
//      H_k = padded half spectrum of slice k written by slice_fft_fwd_kernel.  Output goes
//      straight into the caller's ragged bucket tensors [row][bin][slice][M] (any strides, M contiguous).
//  bins_inv_kernel  (reference: nsgt/nsigtf.py:29-33, :82-92)
//      T_k[coff_j + m'] = DFT_M( (-1)^n c_j[k, n] )[m'] * wi'_j[m'],  wi_j = gd_j M_j (-1)^(pos_j/2)
//      T is the packed [sum_M] row consumed by slice_fft_inv_kernel's gather.
//
// One launch covers all buckets: CTA `blockIdx.x` is job #i of some bucket (binary search in the
// per-launch job table) and owns a contiguous range of (row,slice) units of that bucket.
#include "slicq_fft_tile.cuh"

namespace {

SLICQ_DEVFN int find_bucket(const SlicqBinsParams& p, int job) {
    int lo = 0, hi = p.n_buckets - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (p.b[mid].job_start <= job) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// MG: mask-gradient epilogue of the analysis, OVR: overflow over several runs in the synthesis (see slicq_fft_tile.cuh)
template <int M, int KIND, int A, int B, bool SYNTH, bool MG, bool OVR> struct JobRunner;
template <int M, int A, int B, bool MG, bool OVR> struct JobRunner<M, 1, A, B, false, MG, OVR> {
    static SLICQ_DEVFN void run(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, unsigned char* sm) {
        ana_single<M, MG>(p, b, j, reinterpret_cast<float2*>(sm));
    }
};
template <int M, int A, int B, bool MG, bool OVR> struct JobRunner<M, 1, A, B, true, MG, OVR> {
    static SLICQ_DEVFN void run(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, unsigned char* sm) {
        syn_single<M>(p, b, j, reinterpret_cast<float2*>(sm));
    }
};
template <int M, int A, int B, bool MG, bool OVR> struct JobRunner<M, 2, A, B, false, MG, OVR> {
    static SLICQ_DEVFN void run(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, unsigned char* sm) {
        ana_two_pass<M, A, B, MG>(p, b, j, reinterpret_cast<float2*>(sm));
    }
};
template <int M, int A, int B, bool MG, bool OVR> struct JobRunner<M, 2, A, B, true, MG, OVR> {
    static SLICQ_DEVFN void run(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, unsigned char* sm) {
        syn_two_pass<M, A, B, OVR>(p, b, j, reinterpret_cast<float2*>(sm));
    }
};
template <int M, int A, int B, bool MG, bool OVR> struct JobRunner<M, 3, A, B, false, MG, OVR> {
    static SLICQ_DEVFN void run(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, unsigned char* sm) {
        ana_prime<M, A, B, MG>(p, b, j, reinterpret_cast<float*>(sm));
    }
};
template <int M, int A, int B, bool MG, bool OVR> struct JobRunner<M, 3, A, B, true, MG, OVR> {
    static SLICQ_DEVFN void run(const SlicqBinsParams& p, const SlicqBucketArg& b, const JobCtx& j, unsigned char* sm) {
        syn_prime<M, A, B, OVR>(p, b, j, reinterpret_cast<float*>(sm));
    }
};

template <bool SYNTH, bool MG, bool OVR>
SLICQ_DEVFN void bins_body(const SlicqBinsParams& p, unsigned char* smem) {
    const int job = blockIdx.x;
    const int bi = find_bucket(p, job);
    const SlicqBucketArg& b = p.b[bi];
    JobCtx j;
    j.u0 = (job - b.job_start) * b.units_per_job;
    j.u1 = j.u0 + b.units_per_job;
    if (j.u1 > p.n_rs) j.u1 = p.n_rs;
    if (j.u0 >= j.u1) return;
    j.F = b.n_bins; j.gt = b.gt; j.first_bin = b.first_bin; j.rs0 = p.rs0; j.S = p.S; j.x_rows = SYNTH ? p.x_rows : 0;
    j.aux = SYNTH ? (b.mptr != nullptr) : (b.nptr != nullptr);
    if (SYNTH) {
        // positions of the T planes that no bin covers: zero them for this job's units (see SlicqDeviceTables)
        const int nu = j.u1 - j.u0;
        for (int t = threadIdx.x; t < nu * b.gap_n; t += blockDim.x) {
            const int u = t / b.gap_n, e = t - u * b.gap_n;
            const int2 g = __ldg(p.t.gaps + b.gap_first + e);
            float2* o = p.spec + (long long)(j.u0 + u) * p.spec_stride + g.x;
            for (int c = 0; c < g.y; ++c) o[c] = make_float2(0.f, 0.f);
        }
    }
    switch (b.M) {
#define SLICQ_FFT_SIZE(M_, K_, A_, B_, C_) \
    case M_: JobRunner<M_, K_, A_, B_, SYNTH, MG, OVR>::run(p, b, j, smem); break;
#include "fft_sizes.inc"
#undef SLICQ_FFT_SIZE
        default: break;
    }
}

// resident CTAs per SM the kernels are compiled for: caps a thread at 65536 / (3 * 256) = 85 registers
constexpr int kBinsMinBlocks = 3;

}  // namespace

__global__ void __launch_bounds__(kBinsThreads, kBinsMinBlocks) bins_fwd_kernel(const __grid_constant__ SlicqBinsParams p) {
    SLICQ_DYN_SMEM(unsigned char, smem);
    bins_body<false, false, false>(p, smem);
}

// the analysis with the mask-gradient epilogue (SlicqBinsParams::mask_grad): the adjoint-of-synthesis plan's
// slicq_forward_mask_grad
__global__ void __launch_bounds__(kBinsThreads, kBinsMinBlocks) bins_fwd_mask_grad_kernel(const __grid_constant__ SlicqBinsParams p) {
    SLICQ_DYN_SMEM(unsigned char, smem);
    bins_body<false, true, false>(p, smem);
}

__global__ void __launch_bounds__(kBinsThreads, kBinsMinBlocks) bins_inv_kernel(const __grid_constant__ SlicqBinsParams p) {
    SLICQ_DYN_SMEM(unsigned char, smem);
    bins_body<true, false, false>(p, smem);
}

// the synthesis for plans whose two-pass or prime bins divert more than their first run of outputs to the overflow slot
// (slicq_plan::ov_multi_run: the lowest bins of some Bark / mel filterbanks with few bins or a low fmin)
__global__ void __launch_bounds__(kBinsThreads, kBinsMinBlocks) bins_inv_ovr_kernel(const __grid_constant__ SlicqBinsParams p) {
    SLICQ_DYN_SMEM(unsigned char, smem);
    bins_body<true, false, true>(p, smem);
}

namespace {
template <auto K> int launch_bins(const SlicqBinsParams* p, int n_jobs, int smem_bytes, cudaStream_t s) {
    if (slicq_smem_opt_in<K>(100 * 1024)) return -3;
    SLICQ_LAUNCH(K, dim3(n_jobs), dim3(kBinsThreads), smem_bytes, s, *p);
    return (int)cudaGetLastError();
}
}  // namespace

// host-side launcher (called from slicq_api.cu)
extern "C" int slicq_launch_bins(const SlicqBinsParams* p, int n_jobs, int smem_bytes, SlicqBinsKernel k, cudaStream_t s) {
    if (n_jobs <= 0) return 0;
    switch (k) {
        case bins_fwd: return launch_bins<bins_fwd_kernel>(p, n_jobs, smem_bytes, s);
        case bins_fwd_mask_grad: return launch_bins<bins_fwd_mask_grad_kernel>(p, n_jobs, smem_bytes, s);
        case bins_inv: return launch_bins<bins_inv_kernel>(p, n_jobs, smem_bytes, s);
        case bins_inv_ovr: return launch_bins<bins_inv_ovr_kernel>(p, n_jobs, smem_bytes, s);
    }
    return -2;
}
