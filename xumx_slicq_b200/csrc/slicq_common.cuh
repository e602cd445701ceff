// Common definitions for the sliCQT sm_100a kernels.
//
// Build modes:
//   nvcc (product):  real CUDA, sm_100a.
//   g++ -DSLICQ_EMU (tests only): the *same kernel source* is compiled for the host; CTAs run
//       one after the other, each with blockDim.x real OS threads and a barrier standing in
//       for __syncthreads().  The kernels use no warp-level primitives, so this executes the
//       same per-thread code paths as the GPU.  The emulation library is test infrastructure
//       (tests/emu): the product loader never loads it.
#pragma once

#include <stdint.h>
#include <stddef.h>

#ifdef SLICQ_EMU
// ------------------------------------------------------------------ host emulation shim
#include <cmath>
#include <cstdlib>
#include <cstring>
struct float2 { float x, y; };
struct float4 { float x, y, z, w; };
struct int4 { int x, y, z, w; };
struct int2 { int x, y; };
struct double2 { double x, y; };
static inline int2 make_int2(int a, int b) { int2 r; r.x = a; r.y = b; return r; }
static inline int4 make_int4(int a, int b, int c, int d) { int4 r; r.x = a; r.y = b; r.z = c; r.w = d; return r; }
static inline float4 make_float4(float a, float b, float c, float d) { float4 r; r.x = a; r.y = b; r.z = c; r.w = d; return r; }
static inline float2 make_float2(float a, float b) { float2 r; r.x = a; r.y = b; return r; }
struct dim3 { unsigned x, y, z; dim3(unsigned a = 1, unsigned b = 1, unsigned c = 1) : x(a), y(b), z(c) {} };
extern thread_local dim3 threadIdx;
extern dim3 blockIdx, blockDim, gridDim;
extern unsigned char* slicq_emu_smem;
void slicq_emu_sync();                       // CTA barrier between the emulated threads
#include <functional>
void slicq_emu_launch(dim3 grid, dim3 block, const std::function<void()>& body);
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline __attribute__((always_inline))
#define __launch_bounds__(...)
#define __grid_constant__
static inline void __syncthreads() { slicq_emu_sync(); }
template <class T> static inline T __ldg(const T* p) { return *p; }
typedef int cudaError_t;
typedef void* cudaStream_t;
typedef void* cudaEvent_t;
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2 };
static inline int cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = nullptr; return 0; }
static inline int cudaStreamDestroy(cudaStream_t) { return 0; }
static inline int cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = nullptr; return 0; }
static inline int cudaEventDestroy(cudaEvent_t) { return 0; }
static inline int cudaEventRecord(cudaEvent_t, cudaStream_t) { return 0; }
static inline int cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned = 0) { return 0; }
enum { cudaSuccess = 0 };
enum cudaMemcpyKind { cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaMemcpyDeviceToDevice = 3 };
static inline cudaError_t cudaMalloc(void** p, size_t n) { *p = malloc(n ? n : 1); return *p ? 0 : 2; }
static inline cudaError_t cudaFree(void* p) { free(p); return 0; }
static inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, int) { memcpy(d, s, n); return 0; }
static inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t) { memset(d, v, n); return 0; }
static inline cudaError_t cudaGetLastError() { return 0; }
static inline cudaError_t cudaDeviceSynchronize() { return 0; }
static inline const char* cudaGetErrorString(cudaError_t) { return "emu"; }
static inline cudaError_t cudaSetDevice(int) { return 0; }
static inline cudaError_t cudaGetDevice(int* d) { *d = 0; return 0; }
#define SLICQ_SET_SMEM(kern, bytes) (0)
#define SLICQ_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(slicq_emu_smem)
#define SLICQ_LAUNCH(kern, grid, block, smem, stream, ...) \
    slicq_emu_launch((grid), (block), [&]() { kern(__VA_ARGS__); })
#else
// ------------------------------------------------------------------ real CUDA
#include <cuda_runtime.h>
#define SLICQ_SET_SMEM(kern, bytes) \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))
#define SLICQ_DYN_SMEM(type, name)                                   \
    extern __shared__ __align__(16) unsigned char slicq_smem_raw_[]; \
    type* name = reinterpret_cast<type*>(slicq_smem_raw_)
#define SLICQ_LAUNCH(kern, grid, block, smem, stream, ...) \
    kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif

#define SLICQ_DEVFN __device__ __forceinline__

// ---------------------------------------------------------------------------------------
// fire-and-forget additions to global memory (no return value, performed at L2): the odd slices of the
// synthesis add into samples an even slice has stored, without a read-modify-write round trip
#ifdef SLICQ_EMU
static inline void slicq_red_add(float* p, float v) { *p += v; }
static inline void slicq_red_add2(float* p, float2 v) { p[0] += v.x; p[1] += v.y; }
#else
SLICQ_DEVFN void slicq_red_add(float* p, float v) { asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }
SLICQ_DEVFN void slicq_red_add2(float* p, float2 v) {   // p 8-byte aligned
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
#endif

// ---------------------------------------------------------------------------------------
// asynchronous global -> shared copies (cp.async / LDGSTS): the data lands in shared memory without passing
// through registers, so a phase can have all of its loads in flight at once
#ifdef SLICQ_EMU
static inline void cp_async16(void* d, const void* s) { memcpy(d, s, 16); }
static inline void cp_async8(void* d, const void* s) { memcpy(d, s, 8); }
static inline void cp_async_commit() {}
template <int N> static inline void cp_async_wait() {}
#else
SLICQ_DEVFN void cp_async16(void* d, const void* s) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(d)), "l"(s) : "memory");
}
SLICQ_DEVFN void cp_async8(void* d, const void* s) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(d)), "l"(s) : "memory");
}
SLICQ_DEVFN void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> SLICQ_DEVFN void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
#endif

// ---------------------------------------------------------------------------------------
// bulk asynchronous global -> shared copy (cp.async.bulk, the TMA engine's linear mode) completing on an mbarrier: the
// bytes land in shared memory without passing through the load/store pipe of the SM at all.  dst / src 16-byte aligned,
// bytes a multiple of 16.  One thread arms the barrier and issues the copies; every thread that reads the data waits.
#ifdef SLICQ_EMU
static inline void mbar_init(unsigned long long*, int) {}
static inline void mbar_expect_tx(unsigned long long*, unsigned) {}
static inline void bulk_g2s(void* d, const void* s, unsigned bytes, unsigned long long*) { memcpy(d, s, bytes); }
static inline void mbar_wait(unsigned long long*, unsigned) { slicq_emu_sync(); }   // all threads of the CTA call it
#else
SLICQ_DEVFN void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
SLICQ_DEVFN void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
SLICQ_DEVFN void bulk_g2s(void* d, const void* s, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((unsigned)__cvta_generic_to_shared(d)), "l"(s), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
SLICQ_DEVFN void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}
#endif

// bulk shared -> global copy / float32 reduction (TMA engine, linear mode): the data leaves shared memory without passing
// through registers or the load/store pipe.  Both addresses 16-byte aligned, bytes a multiple of 16.  Shared memory written
// with ordinary stores must be made visible to the async proxy first (fence_proxy_async by the writers, then a barrier);
// the issuing thread keeps the source alive until bulk_wait_read() returns.
#ifdef SLICQ_EMU
static inline void fence_proxy_async() {}
static inline void bulk_s2g(void* g, const void* s, unsigned bytes) { memcpy(g, s, bytes); }
static inline void bulk_s2g_add_f32(void* g, const void* s, unsigned bytes) {
    float* d = static_cast<float*>(g); const float* q = static_cast<const float*>(s);
    for (unsigned i = 0; i < bytes / 4; ++i) d[i] += q[i];
}
static inline void bulk_wait_read() {}
#else
SLICQ_DEVFN void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
SLICQ_DEVFN void bulk_s2g(void* g, const void* s, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(g), "r"((unsigned)__cvta_generic_to_shared(s)), "r"(bytes) : "memory");
}
SLICQ_DEVFN void bulk_s2g_add_f32(void* g, const void* s, unsigned bytes) {
    asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(g), "r"((unsigned)__cvta_generic_to_shared(s)), "r"(bytes) : "memory");
}
SLICQ_DEVFN void bulk_wait_read() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
#endif

// software prefetch of a 128-byte line into L2 (a hint: no register, no scoreboard)
#ifdef SLICQ_EMU
static inline void prefetch_l2(const void*) {}
#else
SLICQ_DEVFN void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
#endif
// the same for a whole 16-byte aligned range with ONE instruction (TMA engine; bytes a multiple of 16)
#ifdef SLICQ_EMU
static inline void bulk_prefetch_l2(const void*, unsigned) {}
#else
SLICQ_DEVFN void bulk_prefetch_l2(const void* p, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
#endif

#define SLICQ_MAX_BUCKETS 96
#define SLICQ_MAX_M 292
// threads of a bins-kernel CTA (k_bins.cu); the plan sizes each bucket's units per iteration to fill them
constexpr int kBinsThreads = 256;

// ---------------------------------------------------------------------------------------
// complex helpers
SLICQ_DEVFN float2 cmul(float2 a, float2 b) {
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
SLICQ_DEVFN float2 cmul_conj(float2 a, float2 b) {  // a * conj(b)
    return make_float2(fmaf(a.x, b.x, a.y * b.y), fmaf(a.y, b.x, -a.x * b.y));
}
SLICQ_DEVFN float2 cconj(float2 a) { return make_float2(a.x, -a.y); }
// Mask-gradient epilogue of the analysis (SlicqBinsParams::mask_grad, slicq_forward_mask_grad): the transform output c is
// S^T g of an output row of the masked synthesis; instead of c the kernel stores d loss / d mask = Re(conj(X) c), X the
// mixture coefficient that row's mask multiplied.  The mixture is only read.
SLICQ_DEVFN float mask_grad_of(float2 x, float2 c) { return fmaf(x.x, c.x, x.y * c.y); }

// ---------------------------------------------------------------------------------------
// mirrored-bin pass of the reference (nsigtf.py:63-80) for a bin that reaches below DC: one entry per spectrum position.
// The entries of one mirrored bin are consecutive, entry first + f for spectrum position f = 0 .. count - 1.
struct SlicqMirrorEntry { int m_src; float weight; };
struct SlicqMirrorBin { int bucket, f_in_bucket, first, count; };

// device-side tables owned by the plan (all in global memory, < 1 MB, L2 resident)
struct SlicqDeviceTables {
    int L;          // slice length (sl_len)
    int N2;         // L / 2 : length of the complex FFT used for the real slice FFT
    int hop;        // L / 2 : slice advance (50 % overlap)
    int n_bins;     // J   (263)
    int n_buckets;  // 70
    int sum_M;      // 18640 coefficients per (row, slice)
    int pad_l;      // spectrum rows carry pad_l mirrored bins below DC ...
    int pad_r;      // ... and pad_r mirrored bins above Nyquist (bins never need reflection logic)
    int tw_lo, tw_hi;       // support of the slicing window: tukey[p] != 0 only for p in [tw_lo, tw_hi)
    int adjoint;            // bit 0: analysis kernels compute the adjoint of the synthesis; bit 1: synthesis kernels that of
                            // the analysis (include/slicq.h SLICQ_PLAN_ADJOINT_OF_*)
    float spec_scale;       // factor on the slice spectrum (1, or 2/L in adjoint mode) ...
    float ends_scale;       // ... and on its DC / Nyquist bins (1, or 1/L)
    const float* tukey;     // [L]   slicing window
    // windows are stored in *centred* order m' = m~ + M/2 (m~ in [-M/2, M/2) the offset from pos_j)
    const float* wf;        // [sum_M] analysis windows  g_j * (-1)^(pos_j/2) / M_j
    const float* wi;        // [sum_M] synthesis windows gd_j * M_j * (-1)^(pos_j/2)
    const int* bin_pos;     // [J]  centre position (rfbas_j)
    const int* bin_M;       // [J]
    const int* bin_coff;    // [J]  offset of bin j inside a packed [sum_M] row
    const float2* post_tw;  // [N2/2 + 1]  exp(-2 pi i k / L)
    const float2* tw;       // concatenated per-bucket twiddles exp(-2 pi i j / M_b), j in [0, M_b)
    // synthesis intermediate T, one row per unit: [plane 0][plane 1][overflow].  Plane q holds the windowed spectra
    // of the bins j with j % 2 == q at their spectrum positions (index pl_off + f); where a bin overlaps earlier bins of
    // its plane, its leading part (up to all of it) goes to the overflow area instead, and the positions no bin of a
    // plane writes ("gaps") are zero-filled by the bins kernel.
    int pl_off, pl_len;           // plane q starts at q * pl_len; position f sits at q * pl_len + pl_off + f  (both even)
    int t_stride;                 // complex elements per row of T (even)
    const int* bin_toff;          // [J] offset in the row of coefficient m' = 0 of bin j
    const int* bin_ov;            // [J] leading coefficients of bin j that go to the overflow area (even, usually 0)
    const int* bin_ovoff;         // [J] offset in the row of the overflow slot of m' = 0
    const int4* ex;               // [n_ex] {f, off0, off1 or -1, fold | round << 1}: position f also receives T[off0]
                                  // (+ T[off1]), conjugated if fold (adjoint of the analysis: overflow below DC / above
                                  // Nyquist); the entries of one round have distinct f
    int n_ex;
    int ex_rounds;                // rounds of the direct and of the folded entries (at most); 1 for most plans
    const int2* gaps;             // {offset in the row, count}: zero-filled per unit by the job of the owning bucket
    // generic slice kernels (k_slice_generic.cu): prime factors of N2 and exp(-2 pi i k / N2)
    int n_fac;
    int fac[20];
    const float2* wN;
    const double2* wP;            // exp(-2 pi i k / fac[0]) in double when the largest factor is > 32 (direct sums of many terms)
    const SlicqMirrorEntry* mir;  // [n_mir]
    int n_mir;                    // 0: no mirrored-bin pass
    const SlicqMirrorBin* mir_bins;   // [n_mir_bins] in bin order
    int n_mir_bins;
    int mir_nf;                   // spectrum positions 0 .. mir_nf - 1 receive mirrored terms (largest count)
    int mir_nc;                   // coefficients of all mirrored bins (sum of their M)
};

// one bucket as a kernel sees it for one call (pointer + strides of the caller's tensor)
struct SlicqBucketArg {
    float2* ptr;          // base of the bucket tensor (complex64 elements)
    long long s_row;      // element stride between rows   (flattened batch*channel)
    long long s_bin;      // element stride between bins
    long long s_slice;    // element stride between slices ; M is contiguous (stride 1)
    int M;
    int first_bin;
    int n_bins;
    int gt;               // (row,slice) units processed concurrently by one CTA iteration
    int tw_off;           // offset into SlicqDeviceTables::tw
    int job_start;        // first job (CTA) index of this bucket inside the launch
    int n_jobs;           // CTAs working on this bucket
    int units_per_job;    // multiple of gt
    int gap_first, gap_n;  // synthesis: entries of SlicqDeviceTables::gaps this bucket zero-fills
    // fused mask*mix synthesis (slicq_inverse_masked): fp32 mask of the same logical shape as the
    // OUTPUT rows [targets*rows][F][S][M]; null = plain synthesis
    const float* mptr;
    // fused magnitude (slicq_forward_norm, reference: ComplexNorm transforms.py:181-208 /
    // abs_of_real_complex phase.py:116-118): analysis also writes |c| as fp32 [rows][F][S][M]; null = off.
    // Mask-gradient analysis (SlicqBinsParams::mask_grad): the fp32 mask gradient [targets*rows][F][S][M]
    float* nptr;
    long long ms_row, ms_bin, ms_slice;   // element strides of the mask (synthesis) / magnitude or mask gradient (analysis)
};

struct SlicqBinsParams {
    SlicqDeviceTables t;
    float2* spec;          // analysis: padded half spectra H [n_rs][spec_stride] ; synthesis: packed T [n_rs][spec_stride]
    long long spec_stride;
    int n_rs;              // (row,slice) units in this chunk
    int rs0;               // flattened index (row * S + slice) of the first unit of the chunk
    int S;                 // slices per row in this call
    int n_buckets;
    int x_rows;            // masked synthesis / mask-gradient analysis: rows of the mixture tensor (output row r reads
                           // mixture row r % x_rows); else 0
    int k0;                // global index of local slice 0 (slice parity for the mirrored-bin pass)
    int mask_grad;         // analysis: b[].ptr is the mixture (read only), b[].nptr receives Re(conj(mixture) c) instead of c
                           // (slicq_forward_mask_grad); 0 = normal analysis
    SlicqBucketArg b[SLICQ_MAX_BUCKETS];
};

struct SlicqSliceParams {
    SlicqDeviceTables t;
    // forward: x = input signal rows ; inverse: y = output signal rows (same fields)
    float* x;
    long long x_row_stride;
    long long T;           // valid samples per row (forward: input length, inverse: output length)
    long long t0;          // global sample index of x[.,0] / y[.,0]
    long long k0;          // global slice index of local slice 0
    float2* spec;          // forward: H out ; inverse: T in
    long long spec_stride;
    float* halo_out;       // inverse: [rows][hop] or null; first half of local slice 0 when k0 > 0
    int n_rs, rs0, S;
    int parity;            // inverse: this launch handles slices with (k & 1) == parity ...
    int par_cs, par_base;  // ... one CTA each: par_cs = such slices per row, par_base = how many precede unit rs0 (set by the launcher)
};

// The long bin: the Nyquist bin of a filterbank band-limited by fmax < fs / 2 is as long as the band between fmax and fs / 2
// (M > SLICQ_MAX_M).  It is the plan's last bucket, a bucket of one bin that the bins kernels skip; long_bin_fwd_kernel /
// long_bin_inv_kernel (k_slice_generic.cu) transform it, one CTA per unit, in shared memory with the generic slice
// kernels' Stockham engine, and do the gap zero-fill of its bucket.  The tables are the plan's; the rest is set per launch.
struct SlicqLongBinParams {
    int M;
    int hoff;              // analysis: offset in a row of H of the bin's first coefficient (m' = 0): pad_l + pos - M / 2
    int toff, ov, ovoff;   // synthesis: offset in a row of T of m' = 0, leading coefficients that go to the overflow slot,
                           // offset of that slot
    int n_fac;
    int fac[20];           // prime factors of M, largest first
    const float2* wM;      // [M] exp(-2 pi i k / M)
    const double2* wP;     // exp(-2 pi i k / fac[0]) in double when fac[0] > 32
    const float* w;        // [M] the bin's window in centred order: wf (analysis) or wi (synthesis)
    const int2* gaps;      // synthesis: the T positions no bin writes that this bucket zero-fills ...
    int gap_n;             // ... (entries)
    float2* spec;          // as SlicqBinsParams
    long long spec_stride;
    int n_rs, rs0, S, x_rows, mask_grad;
    SlicqBucketArg b;      // the caller's view of the bucket
};

// ---------------------------------------------------------------------------------------
// host-side launcher helpers (k_bins.cu, k_slice.cu, k_slice_generic.cu)
#include <atomic>
#include <mutex>

// the four variants of the bins kernel (k_bins.cu)
enum SlicqBinsKernel { bins_fwd, bins_fwd_mask_grad, bins_inv, bins_inv_ovr };

// Opts kernel K in to `bytes` of dynamic shared memory on the current device (the attribute is per device).  The largest
// value set so far is recorded per device; a call that needs no more returns at once, the others set the attribute under
// a lock, so that the attribute only ever rises, also when threads of plans of different lengths race.  0 on success.
template <auto K>
static int slicq_smem_opt_in(int bytes) {
    static std::atomic<int> done[64];
    static std::mutex m;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1;
    std::atomic<int>* rec = (dev >= 0 && dev < 64) ? &done[dev] : nullptr;   // devices beyond the 64th: set every time
    if (rec && rec->load(std::memory_order_acquire) >= bytes) return 0;
    std::lock_guard<std::mutex> lock(m);
    if (rec && rec->load(std::memory_order_relaxed) >= bytes) return 0;
    if (SLICQ_SET_SMEM(K, bytes) != cudaSuccess) return -1;
    if (rec) rec->store(bytes, std::memory_order_release);
    return 0;
}

// The inverse slice kernels run one launch per slice parity, one CTA per slice k with (k & 1) == p.parity among the
// units [rs0, rs0 + n_rs) of rows of S slices.  Sets par_cs (such slices per row) and par_base (how many precede unit rs0)
// in `sp` (a copy of p) and returns the number of CTAs, 0 if there are none.
static inline unsigned slicq_parity_ctas(const SlicqSliceParams& p, SlicqSliceParams& sp) {
    const int S = p.S, q = p.parity, cs = (S + 1 - q) / 2;
    auto count = [&](long long u) { return (u / S) * cs + ((u % S) + 1 - q) / 2; };
    const long long c0 = count(p.rs0), c1 = count((long long)p.rs0 + p.n_rs);
    sp = p;
    sp.par_cs = cs; sp.par_base = (int)c0;
    return c1 > c0 ? (unsigned)(c1 - c0) : 0u;
}
