/* rkfd_engine.cu - sm_100a kernels + device engine of the batched RoKi-FD step path.
 *
 * Kernel rkfd_step_kernel: one thread = one environment (reference rkFDUpdate for one rkFD,
 * src/rkfd_sim.c:560-566); the five dynamics evaluations and the Runge-Kutta-Gill combination of a
 * step are fused in one launch, `nsteps` steps per launch.  Model tables in __constant__ memory
 * (warp-uniform operands), per-env state as env-fastest structure-of-arrays in HBM (every access
 * is a fully coalesced 256-byte warp request), inter-pass link data in a shared-memory column per
 * thread.  fp64 throughout (the reference is double precision).
 */
#include "rkfd_engine.h"

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>

#include "rkfd_kernel.cuh"
#include "rkfd_kin.cuh"
#include "rkfd_model.h"

namespace rkfd {


void cuda_check(int err, const char *what)
{
  if( err != (int)cudaSuccess ){
    char buf[512];
    std::snprintf(buf, sizeof buf, "rokifd_b200: %s failed: %s", what, cudaGetErrorString((cudaError_t)err));
    throw std::runtime_error(buf);
  }
}
#define CK(x) cuda_check((int)(x), #x)

int device_count(){ int n = 0; if( cudaGetDeviceCount(&n) != cudaSuccess ) return 0; return n; }

/* env-major host layout [B][n] <-> device SoA [n][ld]: transposes through a shared-memory tile of TE environments
 * (TE*n contiguous doubles on the env-major side, n rows of TE contiguous doubles on the SoA side), so that both the
 * global loads and the global stores of a warp are contiguous (round 1 moved one env-major row per thread: stride n*8 B,
 * 64 us per array of 262,144 x 7; HBM-bound now: 2 x 14.7 MB per array).  The tile row stride is padded to an odd number
 * of doubles so that the transposed shared-memory accesses spread over the banks. */
constexpr int XP_THREADS = 256, XP_MAXCOL = 128;
/* environments per tile: 64 (512-byte rows on the SoA side) while the tile stays under the 48 KB default limit */
static inline int xp_te(int n){ int te = 64; while( te > 4 && (size_t)te*(n | 1)*sizeof(double) > 40*1024 ) te >>= 1; return te; }
/* columns c0..c0+n-1 of env-major rows of length nrow (wide arrays - the 2,103 contact columns of mighty.ztk - go through in
 * column blocks of XP_MAXCOL) */
__global__ void __launch_bounds__(XP_THREADS) rkfd_scatter_kernel(const double * __restrict__ src, double * __restrict__ dst, int B, int n, int ld, int XP_TE, int nrow, int c0, const int * __restrict__ perm)
{
  extern __shared__ double xp_tile[];
  const int e0 = blockIdx.x*XP_TE, ne = min(XP_TE, B - e0), ns = n | 1;
  for(int i=threadIdx.x; i<ne*n; i+=XP_THREADS){ const int e = i/n, k = i - e*n; xp_tile[e*ns + k] = src[(size_t)(perm ? perm[e0 + e] : e0 + e)*nrow + c0 + k]; }
  __syncthreads();
  for(int i=threadIdx.x; i<n*XP_TE; i+=XP_THREADS){ const int k = i/XP_TE, e = i - k*XP_TE; if( e < ne ) dst[(size_t)(c0 + k)*ld + e0 + e] = xp_tile[e*ns + k]; }
}
__global__ void __launch_bounds__(XP_THREADS) rkfd_gather_kernel(const double * __restrict__ src, double * __restrict__ dst, int B, int n, int ld, int XP_TE, int nrow, int c0, const int * __restrict__ perm)
{
  extern __shared__ double xp_tile[];
  const int e0 = blockIdx.x*XP_TE, ne = min(XP_TE, B - e0), ns = n | 1;
  for(int i=threadIdx.x; i<n*XP_TE; i+=XP_THREADS){ const int k = i/XP_TE, e = i - k*XP_TE; if( e < ne ) xp_tile[e*ns + k] = src[(size_t)(c0 + k)*ld + e0 + e]; }
  __syncthreads();
  for(int i=threadIdx.x; i<ne*n; i+=XP_THREADS){ const int e = i/n, k = i - e*n; dst[(size_t)(perm ? perm[e0 + e] : e0 + e)*nrow + c0 + k] = xp_tile[e*ns + k]; }
}
static void xp_scatter(const double *src, double *dst, int B, int n, int ld, cudaStream_t st, const int *perm)
{
  for(int c0=0; c0<n; c0+=XP_MAXCOL){ const int nc = n - c0 < XP_MAXCOL ? n - c0 : XP_MAXCOL, te = xp_te(nc);
    rkfd_scatter_kernel<<<(B + te - 1)/te, XP_THREADS, (size_t)te*(nc | 1)*sizeof(double), st>>>(src, dst, B, nc, ld, te, n, c0, perm); }
}
static void xp_gather(const double *src, double *dst, int B, int n, int ld, cudaStream_t st, const int *perm)
{
  for(int c0=0; c0<n; c0+=XP_MAXCOL){ const int nc = n - c0 < XP_MAXCOL ? n - c0 : XP_MAXCOL, te = xp_te(nc);
    rkfd_gather_kernel<<<(B + te - 1)/te, XP_THREADS, (size_t)te*(nc | 1)*sizeof(double), st>>>(src, dst, B, nc, ld, te, n, c0, perm); }
}

/* ---- environment re-sort ----------------------------------------------------------------------------------------
 * Environments never interact and the kernels address them by SLOT (thread index), so the engine is free to choose which
 * environment lives in which slot.  Every `resort interval` steps it orders the slots by the number of active contact
 * vertices (descending): the 32 lanes of a warp then hold environments with the same amount of contact work - the penalty
 * force code runs with full warps instead of 7 of 32 lanes, warps (and whole blocks) without contacts skip it and its
 * barriers, and the rigid-contact solvers find their environments packed into few warps.  Results per environment do not
 * depend on the slot (bit-identical).  perm[slot] = environment, inv[environment] = slot; the host-side API maps through
 * them in the transposing copies. */
constexpr int SORT_BINS = 256;     /* keys are bytes; the sort kernels run 256 threads per block */
__global__ void __launch_bounds__(256) rkfd_sort_key_kernel(const unsigned long long * __restrict__ cflags, const unsigned char * __restrict__ work, int nfw, int ld, int B, unsigned char *key, int *bins)
{
  __shared__ int h[SORT_BINS];
  if( threadIdx.x < SORT_BINS ) h[threadIdx.x] = 0;
  __syncthreads();
  const int sl = blockIdx.x*blockDim.x + threadIdx.x;
  if( sl < B ){
    int na = 0;
    for(int w=0;w<nfw;w++) na += __popcll(cflags[(size_t)w*ld + sl] & 0x5555555555555555ull);
    /* worlds under the Vert / Volume solver: the work class of the environment's last rigid solve (contacts or pairs x
     * active-set iterations, written by the step kernel) - the lanes of a warp then leave the active-set loop together */
    if( work && work[sl] ) na = work[sl];
    if( na > SORT_BINS-1 ) na = SORT_BINS-1;
    key[sl] = (unsigned char)na; atomicAdd(&h[na], 1);
  }
  __syncthreads();
  if( threadIdx.x < SORT_BINS && h[threadIdx.x] ) atomicAdd(&bins[threadIdx.x], h[threadIdx.x]);
}
/* first slot of every bin, most contacts first */
__global__ void rkfd_sort_offsets_kernel(int *bins){ if( threadIdx.x == 0 ){ int run = 0; for(int k=SORT_BINS-1;k>=0;k--){ const int c = bins[k]; bins[k] = run; run += c; } } }
__global__ void __launch_bounds__(256) rkfd_sort_assign_kernel(const unsigned char * __restrict__ key, int *cursor, int *newpos, int B)
{
  /* one atomic per (warp, bin): lanes with the same key take consecutive slots in lane order */
  const int sl = blockIdx.x*blockDim.x + threadIdx.x; const unsigned lane = threadIdx.x & 31;
  const int k = sl < B ? (int)key[sl] : -1;
  const unsigned peers = __match_any_sync(0xffffffffu, k);
  int base = 0;
  if( k >= 0 && lane == (unsigned)(__ffs(peers) - 1) ) base = atomicAdd(&cursor[k], __popc(peers));
  base = __shfl_sync(0xffffffffu, base, __ffs(peers) - 1);
  if( k >= 0 ) newpos[sl] = base + __popc(peers & ((1u << lane) - 1u));
}
template <class T> __global__ void __launch_bounds__(256) rkfd_permute_rows_kernel(const T * __restrict__ src, T * __restrict__ dst, const int * __restrict__ newpos, int B, int nrows, int ld)
{
  const int sl = blockIdx.x*blockDim.x + threadIdx.x;
  if( sl >= B ) return;
  const int d = newpos[sl];
  for(int r=0;r<nrows;r++) dst[(size_t)r*ld + d] = src[(size_t)r*ld + sl];
}
__global__ void __launch_bounds__(256) rkfd_perm_compose_kernel(const int * __restrict__ perm_old, const int * __restrict__ newpos, int *perm_new, int *inv_new, int B)
{
  const int sl = blockIdx.x*blockDim.x + threadIdx.x;
  if( sl >= B ) return;
  const int e = perm_old ? perm_old[sl] : sl, d = newpos[sl];
  perm_new[d] = e; inv_new[e] = d;
}

/* ---- environment reset -------------------------------------------------------------------------------------------
 * The committing evaluation of rkFDUpdateInit for a list of environments that sit in scattered slots: a launch covers whole
 * blocks, so it cannot run in place without committing the neighbours as well.  The listed environments are gathered into
 * a compact sub-state (slot i = list entry i), evaluated there by the shard's own kernel variant in mode 2, and the rows the
 * re-sort permutes (plus the work class) are scattered back to their slots.  Results per environment do not depend on the
 * slot or on the other environments of the launch, so an environment comes out exactly as a new engine started from the
 * same state would have it.  The padding slots [n, ld) of the sub-state hold the zero state, like those of a shard. */
constexpr int RESET_CHUNK = 65536;     /* sub-state capacity: longer lists run in chunks */
constexpr int RESET_SEGS = 11, RESET_ROWS = 32;
/* q, q' and u of the sub-state: the given rows, u from the environment's slot when none is given, zero on padding slots; the
 * external wrench (nfx rows) always from the environment's slot: a reset does not change the input.  So do the mass properties
 * (nmr rows), and padding slots take slot 0's: valid values, a padding thread runs the articulated-body pass too */
__global__ void __launch_bounds__(256) rkfd_reset_gather_kernel(StateDev sub, const double * __restrict__ u_cur, int ld, int B, const int * __restrict__ inv,
                                                                const int * __restrict__ envs, int n, const double * __restrict__ q, const double * __restrict__ qd,
                                                                const double * __restrict__ u, int nq, int nl, const double * __restrict__ fext_cur, int nfx,
                                                                const double * __restrict__ mp_cur, int nmr)
{
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if( i >= sub.ld ) return;
  const int e = i < n ? envs[i] : -1;
  const bool live = e >= 0 && e < B;
  const int sl = live ? ( inv ? inv[e] : e ) : 0;
  for(int k=0;k<nq;k++){
    sub.q[0][(size_t)k*sub.ld + i] = live ? q[(size_t)i*nq + k] : 0.0;
    sub.qd[0][(size_t)k*sub.ld + i] = live && qd ? qd[(size_t)i*nq + k] : 0.0;
  }
  for(int k=0;k<nl;k++) sub.u[(size_t)k*sub.ld + i] = !live ? 0.0 : ( u ? u[(size_t)i*nl + k] : u_cur[(size_t)k*ld + sl] );
  for(int k=0;k<nfx;k++) sub.fext[(size_t)k*sub.ld + i] = live ? fext_cur[(size_t)k*ld + sl] : 0.0;
  for(int k=0;k<nmr;k++) sub.mp[(size_t)k*sub.ld + i] = mp_cur[(size_t)k*ld + sl];
}
/* row groups copied back from the sub-state (stride ld_sub, slot i) to the shard (stride ld, the environment's slot) */
struct ResetRows { int nseg; int rows[RESET_SEGS], esz[RESET_SEGS]; const char *src[RESET_SEGS]; char *dst[RESET_SEGS]; };
__global__ void __launch_bounds__(256) rkfd_reset_scatter_kernel(ResetRows rr, const int * __restrict__ envs, int n, int B, const int * __restrict__ inv, int ld_sub, int ld)
{
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if( i >= n ) return;
  const int e = envs[i];
  if( e < 0 || e >= B ) return;
  const int sl = inv ? inv[e] : e;
  /* blockIdx.y: rows [r0, r0 + RESET_ROWS) of the concatenated groups (mighty.ztk has 6,000 rows of anchors and forces) */
  const int r0 = blockIdx.y*RESET_ROWS, r1 = r0 + RESET_ROWS;
  for(int g=0, base=0; g<rr.nseg && base<r1; base+=rr.rows[g], g++){
    const int a = max(r0, base) - base, b = min(r1, base + rr.rows[g]) - base;
    for(int r=a; r<b; r++){
      const size_t si = (size_t)r*ld_sub + i, di = (size_t)r*ld + sl;
      if( rr.esz[g] == 8 ) ((unsigned long long*)rr.dst[g])[di] = ((const unsigned long long*)rr.src[g])[si];
      else if( rr.esz[g] == 4 ) ((unsigned int*)rr.dst[g])[di] = ((const unsigned int*)rr.src[g])[si];
      else rr.dst[g][di] = rr.src[g][si];
    }
  }
}

/* ---- link kinematics (rkFDBatchGetLinkFrames) ---------------------------------------------------------------------
 * One thread per slot walks the links of the table outward (rkfd_kin.cuh) on the committed q, q' (SoA rows: coalesced
 * loads) and keeps the frames that later children need in a shared-memory column per thread.  The outputs are env-major
 * (frame[env][k][12], vel[env][k][6]): every thread puts its rows into a shared-memory tile, and the block then writes the
 * tile environment by environment through perm, as the second half of rkfd_gather_kernel does - each output double is
 * written once, by contiguous warp stores.  The table is a __grid_constant__ parameter: the __constant__ banks belong to the
 * step-kernel variants and to whichever engine uploaded its model last. */
constexpr int KIN_MAX_THREADS = 128;
constexpr size_t KIN_TILE_BYTES = 64*1024;     /* blocks shrink (down to one warp) until tile and keep slots fit in this */
struct KinSrcDev {
  const double *qp, *qdp; const unsigned int *pv; int ld, sl;
  __device__ double q(int k) const { return __ldg(qp + (size_t)k*ld + sl); }
  __device__ double qd(int k) const { return __ldg(qdp + (size_t)k*ld + sl); }
  __device__ unsigned piv() const { return __ldg(pv + sl); }
};
struct KinKeepDev {
  double *col; int nb;
  __device__ double ld(int s, int c) const { return col[(s*KIN_KEEP + c)*nb]; }
  __device__ void st(int s, int c, double v){ col[(s*KIN_KEEP + c)*nb] = v; }
};
struct KinOutDev {
  double *tf, *tv;
  __device__ void frame(int k, int c, double v){ tf[12*k + c] = v; }
  __device__ void vel(int k, int c, double v){ tv[6*k + c] = v; }
};
__global__ void __launch_bounds__(KIN_MAX_THREADS) rkfd_link_frames_kernel(const __grid_constant__ KinDev t, const double * __restrict__ q,
                                                                           const double * __restrict__ qd, const unsigned int * __restrict__ piv,
                                                                           const int * __restrict__ perm, int B, int ld,
                                                                           double * __restrict__ frame, double * __restrict__ vel)
{
  extern __shared__ double kin_smem[];
  const int nb = blockDim.x, tid = threadIdx.x, e0 = blockIdx.x*nb, sl = e0 + tid;
  /* tile rows padded to an odd number of doubles: the lanes of a warp hit different banks */
  const int fw = frame ? 12*t.nsel : 0, vw = vel ? 6*t.nsel : 0, fs = fw ? (fw | 1) : 0, vs = vw ? (vw | 1) : 0;
  double *tf = kin_smem, *tv = tf + (size_t)nb*fs, *keep = tv + (size_t)nb*vs;
  if( sl < B ){
    const KinSrcDev S{q, qd, piv, ld, sl}; KinKeepDev K{keep + tid, nb}; KinOutDev O{tf + (size_t)tid*fs, tv + (size_t)tid*vs};
    kin_walk(t, S, K, O, frame != nullptr, vel != nullptr);
  }
  __syncthreads();
  const int ne = min(nb, B - e0);
  for(int i=tid; i<ne*fw; i+=nb){ const int e = i/fw, c = i - e*fw; frame[(size_t)(perm ? perm[e0 + e] : e0 + e)*fw + c] = tf[e*fs + c]; }
  for(int i=tid; i<ne*vw; i+=nb){ const int e = i/vw, c = i - e*vw; vel[(size_t)(perm ? perm[e0 + e] : e0 + e)*vw + c] = tv[e*vs + c]; }
}

/* rows k0..k0+n-1 of an SoA array <- one value per row, every environment (rkFDChainSetDis/SetVel and
 * rkJointMotorSetInput on a running simulator: the reference's cell windows alias fd->dis/vel, rkfd_sim.c:277-287) */
__global__ void rkfd_fill_rows_kernel(double * __restrict__ dst, int ld, int B, int n, const double * __restrict__ vals)
{
  const int e = blockIdx.x*blockDim.x + threadIdx.x;
  if( e >= B ) return;
  for(int k=0;k<n;k++) dst[(size_t)k*ld + e] = vals[k];
}

/* end-of-run statistics of one shard, reduced on the device (rkFDBatchStats): out[0] environments, [1] environments with an
 * active contact, [2] active contact vertices, [3] environments with a non-zero status word (sums); [4] max |q''|,
 * [5] max |q'| (non-negative doubles order like their bit patterns: atomicMax on the 64-bit integer view) */
__global__ void __launch_bounds__(256) rkfd_stats_kernel(StateDev st, int cur, int nq, int nfw, double *out)
{
  const int e = blockIdx.x*blockDim.x + threadIdx.x;
  double cnt[4] = {0,0,0,0}, mx[2] = {0,0};
  if( e < st.B ){
    int na = 0;
    for(int w=0;w<nfw;w++) na += __popcll(st.cflags[(size_t)w*st.ld + e] & 0x5555555555555555ull);     /* the active bits */
    cnt[0] = 1.0; cnt[1] = na > 0 ? 1.0 : 0.0; cnt[2] = (double)na; cnt[3] = st.status[e] != 0 ? 1.0 : 0.0;
    for(int k=0;k<nq;k++){
      const double a = fabs(st.qdd[(size_t)k*st.ld + e]), v = fabs(st.qd[cur][(size_t)k*st.ld + e]);
      if( a == a && a > mx[0] ) mx[0] = a;
      if( v == v && v > mx[1] ) mx[1] = v;
    }
  }
#pragma unroll
  for(int o=16;o>0;o>>=1){
#pragma unroll
    for(int i=0;i<4;i++) cnt[i] += __shfl_xor_sync(0xffffffffu, cnt[i], o);
#pragma unroll
    for(int i=0;i<2;i++) mx[i] = fmax(mx[i], __shfl_xor_sync(0xffffffffu, mx[i], o));
  }
  if( (threadIdx.x & 31) == 0 ){
    for(int i=0;i<4;i++) if( cnt[i] != 0.0 ) atomicAdd(out + i, cnt[i]);
    for(int i=0;i<2;i++) atomicMax((unsigned long long*)(out + 4 + i), (unsigned long long)__double_as_longlong(mx[i]));
  }
}

/* register-resident DFMA loop on every SM: the measured fp64 roofline denominator (MEASURED_PEAKS.json
 * carries HBM and bf16 only).  8 independent accumulators per thread, 2 flop per DFMA. */
__global__ void __launch_bounds__(256) rkfd_fp64_peak_kernel(double *out, int iters, double a, double b)
{
  double x0 = threadIdx.x*1e-3, x1 = x0+1, x2 = x0+2, x3 = x0+3, x4 = x0+4, x5 = x0+5, x6 = x0+6, x7 = x0+7;
#pragma unroll 1
  for(int i=0;i<iters;i++){
#pragma unroll
    for(int k=0;k<16;k++){
      x0 = fma(x0,a,b); x1 = fma(x1,a,b); x2 = fma(x2,a,b); x3 = fma(x3,a,b);
      x4 = fma(x4,a,b); x5 = fma(x5,a,b); x6 = fma(x6,a,b); x7 = fma(x7,a,b);
    }
  }
  out[blockIdx.x*blockDim.x + threadIdx.x] = x0+x1+x2+x3+x4+x5+x6+x7;
}

double measure_fp64_tflops()
{
  int dev = 0, sms = 0; CK(cudaGetDevice(&dev)); CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int blocks = sms*8, threads = 256, iters = 4096;
  double *out = nullptr; CK(cudaMalloc(&out, (size_t)blocks*threads*sizeof(double)));
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  double best = 0;
  for(int rep=0; rep<5; rep++){
    CK(cudaEventRecord(e0));
    rkfd_fp64_peak_kernel<<<blocks, threads>>>(out, iters, 0.999999, 1e-7);
    CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
    float ms = 0; CK(cudaEventElapsedTime(&ms, e0, e1));
    const double flop = 2.0*8*16*(double)iters*blocks*threads;
    if( rep > 0 && flop/(ms*1e-3)/1e12 > best ) best = flop/(ms*1e-3)/1e12;
  }
  CK(cudaEventDestroy(e0)); CK(cudaEventDestroy(e1)); CK(cudaFree(out));
  return best;
}

struct Shard {
  int dev = 0, e0 = 0, B = 0, ld = 0, cur = 0;
  StateDev st;
  cudaStream_t stream = nullptr; bool own_stream = true;
  double *dstage = nullptr; size_t nstage = 0;
  /* asynchronous transfers: copy streams + a ring of staging buffers, each guarded by a "consumed" event */
  static constexpr int NRING = 8;
  cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
  double *ring[NRING] = {nullptr}; cudaEvent_t ring_done[NRING] = {nullptr}; cudaEvent_t ring_ready[NRING] = {nullptr};
  int ring_next = 0; bool ring_init = false;
  const KernelVariant *kv = nullptr; size_t smem = 0;
  /* environment re-sort: perm[slot] = environment (nullptr: identity), host copies made on demand */
  int *perm = nullptr, *inv = nullptr, *perm_buf[2] = {nullptr, nullptr}, *inv_buf = nullptr, *newpos = nullptr, *bins = nullptr; unsigned char *key = nullptr;
  void *ptmp = nullptr; size_t ptmp_bytes = 0; int perm_cur = 0, steps_since_sort = 0; long long sorts = 0;
  std::vector<int> h_perm; bool h_perm_valid = false;
  /* environment reset (Engine::reset_envs): one buffer for the sub-state of up to rcap environments and the host path's staging */
  char *rbuf = nullptr; int rcap = 0;
  /* link kinematics: the host path's device outputs (allocated on first use, grown when a call needs more) */
  double *kbuf = nullptr; size_t kcap = 0; bool kin_smem_attr = false;
  std::vector<void*> allocs;
};

static int g_next_engine_id = 1;
static int variant_index(const KernelVariant *kv);

template <class T> static T *dalloc(Shard &s, size_t n)
{
  void *p = nullptr; if( n == 0 ) n = 1;
  CK(cudaMalloc(&p, n*sizeof(T))); CK(cudaMemset(p, 0, n*sizeof(T)));
  s.allocs.push_back(p); return (T*)p;
}

/* kernel variants, one translation unit each (rkfd_kernel_variant.cu): BLOCK_GSCR_RIGID_SPEC_MINB */
#define RKFD_VARIANT_LIST(X) \
  X(128,1,1,7,2) X(128,0,1,7,2) X(64,0,1,7,4) X(128,0,0,5,4) X(128,0,0,8,4) X(128,0,0,9,4) X(128,0,0,10,4) X(128,0,0,11,2) X(256,0,0,5,2) X(512,0,0,5,1) X(256,0,0,6,2) X(256,0,0,3,2) X(512,0,0,3,1) X(128,0,0,3,4) X(128,0,0,3,3) X(128,0,0,4,4) X(128,0,0,1,1) X(256,0,0,1,1) X(128,0,0,2,1) \
  X(128,0,0,0,1) X(256,0,0,0,1) X(64,0,0,0,1) X(32,0,0,0,1) X(64,1,0,0,1) \
  X(128,0,1,0,1) X(256,0,1,0,1) X(64,0,1,0,1) X(32,0,1,0,1) X(64,1,1,0,1) X(256,1,1,0,1)
#define RKFD_DECL(B,G,R,S,M) extern const KernelVariant rkfd_variant_##B##_##G##_##R##_##S##_##M;
RKFD_VARIANT_LIST(RKFD_DECL)
#undef RKFD_DECL
/* order = preference among variants that keep the same number of environments resident (measured on B200,
 * profiles/): model specialisations (spec > 0) come first and are taken whenever the model matches; among the
 * tensor-memory specialisations (16 resident warps per SM) the rolled link loops with four 128-thread CTAs per SM
 * are fastest (3.2 k instructions stay in the instruction caches); the fully unrolled code (8.7 k instructions)
 * prefers two 256-thread CTAs (two instruction streams instead of four), one 512-thread CTA loses to barrier stalls */
#define RKFD_REF(B,G,R,S,M) &rkfd_variant_##B##_##G##_##R##_##S##_##M,
static const KernelVariant *g_variants[] = { RKFD_VARIANT_LIST(RKFD_REF) };
#undef RKFD_REF
constexpr int NVARIANTS = (int)(sizeof g_variants / sizeof g_variants[0]);
static int g_model_owner[64][NVARIANTS] = {{0}};   /* [device][variant]: engine whose model sits in that constant bank */

static int variant_index(const KernelVariant *kv){ for(int i=0;i<NVARIANTS;i++) if( g_variants[i] == kv ) return i; return 0; }

Engine::Engine(const ModelDev &model, int B, const std::vector<int> &devices, const double *mp_default) : model_(model), model_tm_(model), B_(B), id_(g_next_engine_id++)
{
  /* the same table with the tensor-memory scratch map, for the generic kernel variant that keeps its T space in TMEM */
  if( !model.has_rigid ) model_layout(model_tm_, true);
  if( B <= 0 ) throw std::runtime_error("rokifd_b200: environment count must be positive");
  if( model.nmp > 0 && !mp_default ) throw std::runtime_error("rokifd_b200: mass properties: the model's own values are needed");
  /* environment re-sort by contact count: every 16 steps when the world has contact pairs (RKFD_RESORT=<steps>, 0: never).
   * Measured on one B200 over 256 settled steps, sorts included (tools/exp_resort.py): C3 0.538 ms per step without, 0.484 /
   * 0.481 / 0.489 / 0.503 ms at 8 / 16 / 32 / 64; C5 MLCP 1.88 -> 1.42, C5 Vert 6.97 -> 5.09 at 16 */
  resort_interval_ = model.npair > 0 ? 16 : 0;
  /* worlds whose step is dominated by a data-dependent rigid solve re-sort more often (the sort costs ~0.1-0.2 ms): under the
   * Volume solver every step (C4, 131,072 envs: 30.3 ms per step at 16, 22.6 at 4, 20.5 at 2, 18.8 at 1), under the Vert QP
   * every 4 (C5: 4.39 -> 4.32 ms) */
  if( model.npair > 0 && model.has_rigid ) resort_interval_ = model.solver == S_VOLUME ? 1 : ( model.solver == S_VERT ? 4 : 16 );
  if( const char *rs = std::getenv("RKFD_RESORT") ) resort_interval_ = std::atoi(rs);
  if( device_count() <= 0 ) throw std::runtime_error("rokifd_b200: no CUDA device (there is no CPU fallback)");
  std::vector<int> devs = devices;
  if( devs.empty() ){ int d = 0; CK(cudaGetDevice(&d)); devs.push_back(d); }
  const int G = (int)devs.size();
  int prev = 0; CK(cudaGetDevice(&prev));
  for(int g=0; g<G; g++){
    /* contiguous env blocks: env e -> shard floor(e*G/B) */
    const int e0 = (int)((long long)B*g/G), e1 = (int)((long long)B*(g+1)/G);
    if( e1 <= e0 ) continue;
    Shard *s = new Shard; shards_.push_back(s);
    s->dev = devs[g]; s->e0 = e0; s->B = e1-e0; s->ld = (s->B + 511) & ~511;   /* whole blocks of any variant (<= 512 threads): no thread exits early */
    CK(cudaSetDevice(s->dev));
    CK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    const int nq = model.nq > 0 ? model.nq : 1, nl = model.nl > 0 ? model.nl : 1, ns = model.nslot > 0 ? model.nslot : 1;
    StateDev &st = s->st; std::memset(&st, 0, sizeof st);
    st.B = s->B; st.ld = s->ld;
    for(int k=0;k<2;k++){ st.q[k] = dalloc<double>(*s, (size_t)nq*s->ld); st.qd[k] = dalloc<double>(*s, (size_t)nq*s->ld); }
    st.qdd = dalloc<double>(*s, (size_t)nq*s->ld);
    st.u = dalloc<double>(*s, (size_t)nl*s->ld);
    st.piv_prev = dalloc<double>(*s, (size_t)nq*s->ld);
    st.piv_type = dalloc<unsigned int>(*s, s->ld);
    st.cflags = dalloc<unsigned long long>(*s, (size_t)(model.nfw > 0 ? model.nfw : 1)*s->ld);
    st.cref = dalloc<double>(*s, (size_t)3*ns*s->ld);
    st.cf = dalloc<double>(*s, (size_t)3*ns*s->ld);
    st.status = dalloc<int>(*s, s->ld);
    st.fext = model.nfext > 0 ? dalloc<double>(*s, (size_t)6*model.nfext*s->ld) : nullptr;     /* zero: the initial wrench */
    st.mp = model.nmp > 0 ? dalloc<double>(*s, (size_t)10*model.nmp*s->ld) : nullptr;          /* filled below */
    st.work = ( std::getenv("RKFD_NO_WORK_SORT") == nullptr && model.has_rigid && model.solver != S_MLCP ) ? dalloc<unsigned char>(*s, s->ld) : nullptr;
    /* per-warp workspace of the dense warp-cooperative contact solve; the single-link paths use ws1 only */
    st.ws = ( model.ws_doubles > 0 && model.rigid_link < 0 ) ? dalloc<double>(*s, (size_t)(s->ld/32)*model.ws_doubles) : nullptr;
    st.ws1 = model.ws1_doubles > 0 ? dalloc<double>(*s, (size_t)model.ws1_doubles*s->ld) : nullptr;
    int nmax = nq; if( nl > nmax ) nmax = nl; if( 3*ns > nmax ) nmax = 3*ns; if( 6*model.nfext > nmax ) nmax = 6*model.nfext;
    if( 10*model.nmp > nmax ) nmax = 10*model.nmp;
    /* the kernels index the per-environment arrays with 32-bit element offsets (row * ld + e) */
    if( (unsigned long long)nmax*(unsigned long long)s->ld >= (1ull << 32) )
      throw std::runtime_error("rokifd_b200: rows x environments per device exceed 2^32 elements - spread the batch over more devices (rkFDBatchSetDevices)");
    s->nstage = (size_t)nmax*s->B; if( s->nstage < 256 ) s->nstage = 256; s->dstage = dalloc<double>(*s, s->nstage);
    if( st.mp ){    /* every slot, the padding [B, ld) too, starts with the model's own mass properties */
      CK(cudaMemcpy(s->dstage, mp_default, (size_t)10*model.nmp*sizeof(double), cudaMemcpyHostToDevice));
      rkfd_fill_rows_kernel<<<s->ld/256, 256>>>(st.mp, s->ld, s->ld, 10*model.nmp, s->dstage);
      CK(cudaGetLastError());
    }
    /* launch configuration: the block size that keeps most environments resident per SM; scratch in HBM
     * (gscr) only when no shared-memory variant fits */
    int best = 0; const bool rigid = model.has_rigid;
    /* model specialisation (RKFD_SPEC=0 forces the generic kernel: tuning / comparison aid) */
    unsigned specs = spec_match_mask(model);
    if( !model.has_rigid && model_tm_.ntspace > 0 && model_tm_.ntspace <= SPEC_GENERIC_TM_MAX_T ) specs |= 1u << SPEC_GENERIC_TM;
    if( const char *fs = std::getenv("RKFD_SPEC") ) specs &= 1u << std::atoi(fs);    /* 0: generic kernel only */
    /* scratch in HBM even when shared memory would fit: tuning aid, and the default of the Volume solver - its lanes live in
     * thread-local memory anyway and the 291-double column of a legged tree leaves room for 2 warps per SM only (C4,
     * 131,072 envs: 130 -> 103 ms per step) */
    const int pass0 = ( std::getenv("RKFD_FORCE_GSCR") || ( model.has_rigid && model.solver == S_VOLUME && !std::getenv("RKFD_FORCE_SMEM") ) ) ? 2 : 0;
    /* Volume solver: one 256-thread block per SM - its phases are separated by block barriers, so that the eight warps of
     * an SM stay inside the same piece of code (C4, 131,072 envs: 68 ms per step with 64-thread blocks, 55 ms with 256) */
    const bool volume = model.has_rigid && model.solver == S_VOLUME;
    for(int attempt = volume ? 0 : 1; attempt < 2 && best == 0; attempt++)
    for(int pass=pass0; pass<3 && best==0; pass++)
      for(const KernelVariant *kv : g_variants){
        if( attempt == 0 && !std::getenv("RKFD_FORCE_BLOCK") && kv->block != 256 ) continue;
        /* pass 0: a matching specialisation; 1: generic, shared-memory scratch; 2: generic, scratch in HBM */
        /* a specialisation may keep its scratch column in HBM: the rigid layout of the 7-joint arm (134 doubles) leaves room
         * for ONE 128-thread block per SM in shared memory, i.e. one warp per scheduler; through L1/L2 two blocks are resident
         * and C5 steps in 1.51 instead of 1.95 ms (MLCP) / 4.85 instead of 5.96 ms (Vert).  RKFD_FORCE_SMEM: shared memory only */
        if( kv->rigid != rigid ) continue;
        if( pass == 0 ? ( kv->gscr && std::getenv("RKFD_FORCE_SMEM") ) : kv->gscr != (pass == 2) ) continue;
        if( pass == 0 ? !( kv->spec > 0 && (specs >> kv->spec & 1u) ) : kv->spec != 0 ) continue;
        if( const char *fb = std::getenv("RKFD_FORCE_BLOCK") ) if( std::atoi(fb) != kv->block ) continue;   /* tuning aids */
        if( const char *fm = std::getenv("RKFD_FORCE_MINB") ) if( std::atoi(fm) != kv->minb ) continue;
        const int nscr = kv->spec == SPEC_GENERIC_TM ? model_tm_.nscratch : ( kv->spec ? spec_nscratch(kv->spec) : model.nscratch );
        size_t smem = kv->gscr ? 0 : (size_t)nscr*kv->block*sizeof(double);
        if( const char *pad = std::getenv("RKFD_SMEM_PAD") ) smem += (size_t)std::atoi(pad);   /* tuning aid: lowers occupancy */
        if( smem > 227*1024 ) continue;
        int nb = kv->blocks_per_sm(smem);
        /* rigid worlds: the first variant of the list that fits (128-thread blocks: C5 with 15 % of the envs in contact
         * steps in 3.7 ms against 5.6 ms with 32-thread blocks although those keep 25 % more threads resident - the
         * 23 k-instruction kernel lives on what its warps share in the instruction cache) */
        if( rigid && best > 0 ) continue;
        if( nb*kv->block > best ){ best = nb*kv->block; s->kv = kv; s->smem = smem; }
      }
    /* generic rigid kernel with a large scratch column (trees: 291 doubles for the biped): shared memory leaves room for one
     * 64-thread block per SM; with the column in HBM four are resident (both soles of the biped on the rigid floor, dense
     * MLCP path: 26.5 -> 14.5 ms per step of 16,384 envs) */
    if( rigid && s->kv && s->kv->spec == 0 && !s->kv->gscr && best < 256 && !std::getenv("RKFD_FORCE_SMEM") && !std::getenv("RKFD_FORCE_BLOCK") )
      for(const KernelVariant *kv : g_variants){
        if( !kv->rigid || !kv->gscr || kv->spec != 0 || kv->block != 64 ) continue;
        const int nb = kv->blocks_per_sm(0);
        if( nb*kv->block >= 2*best ){ best = nb*kv->block; s->kv = kv; s->smem = 0; break; }
      }
    if( s->kv && s->kv->gscr ) st.scratch = dalloc<double>(*s, (size_t)model.nscratch*s->ld);
    if( best == 0 ) throw std::runtime_error("rokifd_b200: no launch configuration fits this model");
    /* the zero-fills above ran on the legacy default stream, which this non-blocking stream does not wait for */
    CK(cudaDeviceSynchronize());
  }
  CK(cudaSetDevice(prev));
}

Engine::~Engine()
{
  int prev = 0; cudaGetDevice(&prev);
  for(Shard *s : shards_){
    cudaSetDevice(s->dev);
    cudaStreamSynchronize(s->stream);
    if( s->kv && g_model_owner[s->dev & 63][variant_index(s->kv)] == id_ ) g_model_owner[s->dev & 63][variant_index(s->kv)] = 0;
    if( s->ring_init ){ cudaStreamSynchronize(s->h2d_stream); cudaStreamSynchronize(s->d2h_stream);
      for(int i=0;i<Shard::NRING;i++){ cudaEventDestroy(s->ring_done[i]); cudaEventDestroy(s->ring_ready[i]); }
      cudaStreamDestroy(s->h2d_stream); cudaStreamDestroy(s->d2h_stream); }
    for(void *p : s->allocs) cudaFree(p);
    cudaFree(s->rbuf); cudaFree(s->kbuf);
    if( s->own_stream && s->stream ) cudaStreamDestroy(s->stream);
    delete s;
  }
  cudaSetDevice(prev);
}

void Engine::upload_model(Shard &s)
{
  int &owner = g_model_owner[s.dev & 63][variant_index(s.kv)];
  if( owner == id_ ) return;
  /* another engine's kernels may still read the constant table on this device */
  if( owner != 0 ) CK(cudaDeviceSynchronize());
  CK(s.kv->upload(s.kv->spec == SPEC_GENERIC_TM ? &model_tm_ : &model_, s.stream));
  owner = id_;
}

/* the shard's step kernel on `st`: the shard's own state, or the sub-state of a reset */
void Engine::launch(Shard &s, const StateDev &st, int cur, int mode, int nsteps)
{
  CK(cudaSetDevice(s.dev));
  upload_model(s);
  s.kv->launch(st, cur, mode, nsteps, (st.ld + s.kv->block - 1)/s.kv->block, s.smem, s.stream);
  CK(cudaGetLastError());
  launches_++;
}

static const std::vector<int> &host_perm(Shard &s)
{
  if( !s.h_perm_valid ){
    s.h_perm.resize(s.B);
    if( s.perm ){ CK(cudaStreamSynchronize(s.stream)); CK(cudaMemcpy(s.h_perm.data(), s.perm, (size_t)s.B*sizeof(int), cudaMemcpyDeviceToHost)); }
    else for(int i=0;i<s.B;i++) s.h_perm[i] = i;
    s.h_perm_valid = true;
  }
  return s.h_perm;
}

void Engine::resort(Shard &s)
{
  const int nq = model_.nq > 0 ? model_.nq : 1, nl = model_.nl > 0 ? model_.nl : 1, ns = model_.nslot > 0 ? model_.nslot : 1, nfw = model_.nfw > 0 ? model_.nfw : 1;
  if( !s.newpos ){
    s.newpos = dalloc<int>(s, s.ld); s.bins = dalloc<int>(s, SORT_BINS); s.key = dalloc<unsigned char>(s, s.ld);
    s.perm_buf[0] = dalloc<int>(s, s.ld); s.perm_buf[1] = dalloc<int>(s, s.ld); s.inv_buf = dalloc<int>(s, s.ld);
    size_t rows = (size_t)3*ns; if( (size_t)nq > rows ) rows = nq; if( (size_t)nl > rows ) rows = nl; if( (size_t)nfw > rows ) rows = nfw;
    if( (size_t)6*model_.nfext > rows ) rows = (size_t)6*model_.nfext;
    if( (size_t)10*model_.nmp > rows ) rows = (size_t)10*model_.nmp;
    s.ptmp_bytes = rows*s.ld*sizeof(double); s.ptmp = dalloc<double>(s, rows*s.ld);
    CK(cudaDeviceSynchronize());       /* dalloc's zero-fill runs on the legacy stream */
  }
  const int grid = (s.ld + 255)/256;
  CK(cudaMemsetAsync(s.bins, 0, SORT_BINS*sizeof(int), s.stream));
  rkfd_sort_key_kernel<<<grid, 256, 0, s.stream>>>(s.st.cflags, s.st.work, nfw, s.ld, s.B, s.key, s.bins);
  rkfd_sort_offsets_kernel<<<1, 32, 0, s.stream>>>(s.bins);
  rkfd_sort_assign_kernel<<<grid, 256, 0, s.stream>>>(s.key, s.bins, s.newpos, s.B);
  CK(cudaGetLastError());
  resort_kernels_ += 4;      /* key, offsets, assign above; the composition of the order below */
  auto perm_rows = [&](void *base, size_t elem, int nrows){
    if( !base || nrows <= 0 ) return;
    resort_kernels_++;
    const size_t bytes = (size_t)nrows*s.ld*elem;
    /* the padding slots [B, ld) keep their (valid, zero-state) content */
    CK(cudaMemcpyAsync(s.ptmp, base, bytes, cudaMemcpyDeviceToDevice, s.stream));
    if( elem == 8 ) rkfd_permute_rows_kernel<unsigned long long><<<grid, 256, 0, s.stream>>>((const unsigned long long*)s.ptmp, (unsigned long long*)base, s.newpos, s.B, nrows, s.ld);
    else rkfd_permute_rows_kernel<unsigned int><<<grid, 256, 0, s.stream>>>((const unsigned int*)s.ptmp, (unsigned int*)base, s.newpos, s.B, nrows, s.ld);
    CK(cudaGetLastError());
  };
  StateDev &st = s.st;
  perm_rows(st.q[s.cur], 8, nq); perm_rows(st.qd[s.cur], 8, nq); perm_rows(st.qdd, 8, nq); perm_rows(st.u, 8, nl); perm_rows(st.fext, 8, 6*model_.nfext); perm_rows(st.mp, 8, 10*model_.nmp);
  perm_rows(st.piv_prev, 8, nq); perm_rows(st.piv_type, 4, 1); perm_rows(st.cflags, 8, nfw);
  perm_rows(st.cref, 8, 3*ns); perm_rows(st.cf, 8, 3*ns); perm_rows(st.status, 4, 1);
  int *pn = s.perm_buf[s.perm_cur ^ 1];
  rkfd_perm_compose_kernel<<<grid, 256, 0, s.stream>>>(s.perm, s.newpos, pn, s.inv_buf, s.B);
  CK(cudaGetLastError());
  s.perm = pn; s.inv = s.inv_buf; s.perm_cur ^= 1; s.h_perm_valid = false; s.steps_since_sort = 0; s.sorts++;
}

/* Shard::rbuf for a reset sub-state of leading dimension ld (a multiple of 512, <= cap): the host path's staging for cap
 * environments (ids, q, q', u), then the rows a new engine holds zero (contiguous: one memset clears them), then q, q', u and
 * the evaluation's workspaces.  With base = 0 it gives the size. */
struct ResetLayout { StateDev st; size_t zero_ofs, zero_bytes, bytes; int *envs; double *q, *qd, *u; };
static ResetLayout reset_layout(const Shard &s, const ModelDev &m, int ld, int cap, char *base)
{
  const size_t nq = m.nq > 0 ? m.nq : 1, nl = m.nl > 0 ? m.nl : 1, ns = m.nslot > 0 ? m.nslot : 1, nfw = m.nfw > 0 ? m.nfw : 1, L = ld, C = cap;
  size_t off = 0;
  auto take = [&](size_t bytes){ void *p = (void*)((uintptr_t)base + off); off += (bytes + 255) & ~(size_t)255; return p; };
  ResetLayout r; std::memset(&r, 0, sizeof r);
  r.envs = (int*)take(4*C); r.q = (double*)take(8*nq*C); r.qd = (double*)take(8*nq*C); r.u = (double*)take(8*nl*C);
  StateDev &st = r.st;
  st.B = ld; st.ld = ld;
  r.zero_ofs = off;
  st.qdd = (double*)take(8*nq*L); st.piv_prev = (double*)take(8*nq*L); st.cflags = (unsigned long long*)take(8*nfw*L);
  st.cref = (double*)take(8*3*ns*L); st.cf = (double*)take(8*3*ns*L);
  st.piv_type = (unsigned int*)take(4*L); st.status = (int*)take(4*L);
  if( s.st.work ) st.work = (unsigned char*)take(L);
  r.zero_bytes = off - r.zero_ofs;
  for(int k=0;k<2;k++){ st.q[k] = (double*)take(8*nq*L); st.qd[k] = (double*)take(8*nq*L); }
  st.u = (double*)take(8*nl*L);
  if( s.st.fext ) st.fext = (double*)take(8*6*(size_t)m.nfext*L);
  if( s.st.mp ) st.mp = (double*)take(8*10*(size_t)m.nmp*L);
  if( s.st.scratch ) st.scratch = (double*)take(8*(size_t)m.nscratch*L);
  if( s.st.ws ) st.ws = (double*)take(8*(L/32)*(size_t)m.ws_doubles);
  if( s.st.ws1 ) st.ws1 = (double*)take(8*(size_t)m.ws1_doubles*L);
  r.bytes = off;
  return r;
}
/* the sub-state for lists of up to n environments (allocated on first use, grown when a longer list comes) */
static int reset_reserve(Shard &s, const ModelDev &m, int n)
{
  const int ld = ((n < RESET_CHUNK ? n : RESET_CHUNK) + 511) & ~511;
  if( ld > s.rcap ){
    CK(cudaStreamSynchronize(s.stream));      /* earlier resets may still use the old buffer */
    CK(cudaFree(s.rbuf)); s.rbuf = nullptr; s.rcap = 0;
    const size_t bytes = reset_layout(s, m, ld, ld, nullptr).bytes;
    CK(cudaMalloc(&s.rbuf, bytes)); CK(cudaMemset(s.rbuf, 0, bytes));
    CK(cudaDeviceSynchronize());              /* the zero fill runs on the legacy stream */
    s.rcap = ld;
  }
  return ld;
}

void Engine::reset_chunk(Shard &s, int n, const int *envs, const double *q, const double *qd, const double *u)
{
  const int nq = model_.nq, nl = model_.nl, ns = model_.nslot > 0 ? model_.nslot : 1, nfw = model_.nfw > 0 ? model_.nfw : 1;
  const int ld = reset_reserve(s, model_, n);
  const ResetLayout r = reset_layout(s, model_, ld, s.rcap, s.rbuf);
  const StateDev &sub = r.st;
  CK(cudaMemsetAsync(s.rbuf + r.zero_ofs, 0, r.zero_bytes, s.stream));
  rkfd_reset_gather_kernel<<<ld/256, 256, 0, s.stream>>>(sub, s.st.u, s.ld, s.B, s.inv, envs, n, q, qd, u, nq, nl, s.st.fext, 6*model_.nfext, s.st.mp, 10*model_.nmp);
  CK(cudaGetLastError());
  launch(s, sub, 0, 2, 0);                    /* rkFDUpdateInit's committing evaluation, on the sub-state */
  ResetRows rr; std::memset(&rr, 0, sizeof rr);
  auto seg = [&](const void *src, void *dst, int rows, int esz){ rr.src[rr.nseg] = (const char*)src; rr.dst[rr.nseg] = (char*)dst; rr.rows[rr.nseg] = rows; rr.esz[rr.nseg] = esz; rr.nseg++; };
  seg(sub.q[0], s.st.q[s.cur], nq, 8); seg(sub.qd[0], s.st.qd[s.cur], nq, 8); seg(sub.qdd, s.st.qdd, nq, 8); seg(sub.u, s.st.u, nl, 8);
  seg(sub.piv_prev, s.st.piv_prev, nq, 8); seg(sub.cflags, s.st.cflags, nfw, 8); seg(sub.cref, s.st.cref, 3*ns, 8); seg(sub.cf, s.st.cf, 3*ns, 8);
  seg(sub.piv_type, s.st.piv_type, 1, 4); seg(sub.status, s.st.status, 1, 4);
  if( s.st.work ) seg(sub.work, s.st.work, 1, 1);
  int rows = 0; for(int g=0; g<rr.nseg; g++) rows += rr.rows[g];
  rkfd_reset_scatter_kernel<<<dim3((n + 255)/256, (rows + RESET_ROWS - 1)/RESET_ROWS), 256, 0, s.stream>>>(rr, envs, n, s.B, s.inv, ld, s.ld);
  CK(cudaGetLastError());
  reset_kernels_ += 3;                        /* zero fill, gather, scatter */
}

void Engine::reset_envs(int si, int n, const int *envs, const double *q, const double *qd, const double *u)
{
  if( si < 0 || si >= (int)shards_.size() ) throw std::runtime_error("rokifd_b200: reset: shard index out of range");
  if( n <= 0 ) return;
  Shard &s = *shards_[si];
  const int nq = model_.nq, nl = model_.nl;
  int prev = 0; CK(cudaGetDevice(&prev)); CK(cudaSetDevice(s.dev));
  for(int c0=0; c0<n; c0+=RESET_CHUNK){
    const int nc = n - c0 < RESET_CHUNK ? n - c0 : RESET_CHUNK;
    reset_chunk(s, nc, envs + c0, q + (size_t)c0*nq, qd ? qd + (size_t)c0*nq : nullptr, u ? u + (size_t)c0*nl : nullptr);
  }
  CK(cudaSetDevice(prev));
}

void Engine::reset_envs_host(int n, const int *envs, const double *q, const double *qd, const double *u)
{
  if( n <= 0 ) return;
  const int nq = model_.nq, nl = model_.nl;
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    /* this shard's part of the list, with local indices, and its rows */
    std::vector<int> ids; std::vector<double> hq, hqd, hu;
    for(int i=0;i<n;i++){
      const int e = envs[i] - s->e0;
      if( e < 0 || e >= s->B ) continue;
      ids.push_back(e);
      hq.insert(hq.end(), q + (size_t)i*nq, q + (size_t)(i+1)*nq);
      if( qd ) hqd.insert(hqd.end(), qd + (size_t)i*nq, qd + (size_t)(i+1)*nq);
      if( u ) hu.insert(hu.end(), u + (size_t)i*nl, u + (size_t)(i+1)*nl);
    }
    CK(cudaSetDevice(s->dev));
    for(int c0=0; c0<(int)ids.size(); c0+=RESET_CHUNK){
      const int nc = (int)ids.size() - c0 < RESET_CHUNK ? (int)ids.size() - c0 : RESET_CHUNK;
      const int ld = reset_reserve(*s, model_, nc);
      const ResetLayout r = reset_layout(*s, model_, ld, s->rcap, s->rbuf);
      /* the staging is reused by the next chunk only after this chunk's kernels (same stream) */
      CK(cudaMemcpyAsync(r.envs, ids.data() + c0, (size_t)nc*sizeof(int), cudaMemcpyHostToDevice, s->stream));
      CK(cudaMemcpyAsync(r.q, hq.data() + (size_t)c0*nq, (size_t)nc*nq*sizeof(double), cudaMemcpyHostToDevice, s->stream));
      if( qd ) CK(cudaMemcpyAsync(r.qd, hqd.data() + (size_t)c0*nq, (size_t)nc*nq*sizeof(double), cudaMemcpyHostToDevice, s->stream));
      if( u ) CK(cudaMemcpyAsync(r.u, hu.data() + (size_t)c0*nl, (size_t)nc*nl*sizeof(double), cudaMemcpyHostToDevice, s->stream));
      reset_chunk(*s, nc, r.envs, r.q, qd ? r.qd : nullptr, u ? r.u : nullptr);
    }
    /* the host vectors are read by the copies: finish before they go out of scope */
    CK(cudaStreamSynchronize(s->stream));
  }
  CK(cudaSetDevice(prev));
}

void Engine::kin_launch(Shard &s, const KinDev &t, double *frame, double *vel)
{
  const size_t fw = 12*(size_t)t.nsel, vw = 6*(size_t)t.nsel;
  const size_t per_env = sizeof(double)*((frame ? (fw | 1) : 0) + (vel ? (vw | 1) : 0) + (size_t)KIN_KEEP*t.nkeep);
  int nb = KIN_MAX_THREADS;
  while( nb > 32 && nb*per_env > KIN_TILE_BYTES ) nb >>= 1;
  const size_t smem = nb*per_env;
  if( smem > 227*1024 ) throw std::runtime_error("rokifd_b200: link frames: the output tile does not fit in shared memory");
  if( smem > 48*1024 && !s.kin_smem_attr ){
    CK(cudaFuncSetAttribute(rkfd_link_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227*1024)); s.kin_smem_attr = true; }
  rkfd_link_frames_kernel<<<(s.B + nb - 1)/nb, nb, smem, s.stream>>>(t, s.st.q[s.cur], s.st.qd[s.cur], s.st.piv_type, s.perm, s.B, s.ld, frame, vel);
  CK(cudaGetLastError());
  kin_kernels_++;
}

void Engine::link_frames(int si, const KinDev &t, double *frame, double *vel)
{
  if( si < 0 || si >= (int)shards_.size() ) throw std::runtime_error("rokifd_b200: link frames: shard index out of range");
  if( t.nsel == 0 || ( !frame && !vel ) ) return;
  int prev = 0; CK(cudaGetDevice(&prev)); CK(cudaSetDevice(shards_[si]->dev));
  kin_launch(*shards_[si], t, frame, vel);
  CK(cudaSetDevice(prev));
}

void Engine::link_frames_host(const KinDev &t, double *frame, double *vel)
{
  if( t.nsel == 0 || ( !frame && !vel ) ) return;
  const size_t fw = 12*(size_t)t.nsel, vw = 6*(size_t)t.nsel;
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    const size_t need = (size_t)s->B*((frame ? fw : 0) + (vel ? vw : 0));
    if( need > s->kcap ){
      CK(cudaStreamSynchronize(s->stream));      /* an earlier call's copies may still read the old buffer */
      CK(cudaFree(s->kbuf)); s->kbuf = nullptr; s->kcap = 0;
      CK(cudaMalloc(&s->kbuf, need*sizeof(double))); s->kcap = need;
    }
    double *df = frame ? s->kbuf : nullptr, *dv = vel ? s->kbuf + ( frame ? (size_t)s->B*fw : 0 ) : nullptr;
    kin_launch(*s, t, df, dv);
    if( frame ) CK(cudaMemcpyAsync(frame + (size_t)s->e0*fw, df, (size_t)s->B*fw*sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if( vel ) CK(cudaMemcpyAsync(vel + (size_t)s->e0*vw, dv, (size_t)s->B*vw*sizeof(double), cudaMemcpyDeviceToHost, s->stream));
  }
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream)); }
  CK(cudaSetDevice(prev));
}

void Engine::step(int nsteps)
{
  if( nsteps <= 0 ) return;
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    if( resort_interval_ > 0 && s->B > 32 && s->steps_since_sort >= resort_interval_ ){      /* one warp: nothing to group */ CK(cudaSetDevice(s->dev)); resort(*s); }
    s->steps_since_sort += nsteps;
    launch(*s, s->st, s->cur, 0, nsteps);
    if( nsteps & 1 ) s->cur ^= 1;
  }
  CK(cudaSetDevice(prev));
}
void Engine::eval(bool ref)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_) launch(*s, s->st, s->cur, ref ? 2 : 1, 0);
  CK(cudaSetDevice(prev));
}
void Engine::sync()
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream));
    if( s->ring_init ){ CK(cudaStreamSynchronize(s->h2d_stream)); CK(cudaStreamSynchronize(s->d2h_stream)); } }
  CK(cudaSetDevice(prev));
}
void Engine::set_stream(void *stream)
{
  if( shards_.size() != 1 ) throw std::runtime_error("rokifd_b200: set_stream needs a single-device engine");
  Shard *s = shards_[0];
  CK(cudaSetDevice(s->dev));
  CK(cudaStreamSynchronize(s->stream));
  if( s->own_stream && s->stream ) CK(cudaStreamDestroy(s->stream));
  s->stream = (cudaStream_t)stream; s->own_stream = false;
}
void Engine::slot_map(int si, int *perm)
{
  if( si < 0 || si >= (int)shards_.size() ) return;
  int prev = 0; CK(cudaGetDevice(&prev)); CK(cudaSetDevice(shards_[si]->dev));
  const std::vector<int> &hp = host_perm(*shards_[si]);
  for(int i=0;i<shards_[si]->B;i++) perm[i] = hp[i];
  CK(cudaSetDevice(prev));
}
long long Engine::resorts() const { long long n = 0; for(const Shard *s : shards_) n += s->sorts; return n; }
void Engine::kernel_variant(int si, int v[5]) const
{
  if( si < 0 || si >= (int)shards_.size() ) throw std::runtime_error("rokifd_b200: kernel variant: shard index out of range");
  const KernelVariant *kv = shards_[si]->kv;
  v[0] = kv->block; v[1] = kv->gscr; v[2] = kv->rigid; v[3] = kv->spec; v[4] = kv->minb;
}
void *Engine::device_ptr(int si, int which, int *ld, int *B)
{
  if( si < 0 || si >= (int)shards_.size() ) return nullptr;
  Shard *s = shards_[si];
  if( ld ) *ld = s->ld; if( B ) *B = s->B;
  switch(which){ case 0: return s->st.q[s->cur]; case 1: return s->st.qd[s->cur]; case 2: return s->st.qdd; case 3: return s->st.u; default: return nullptr; }
}

/* ---- host <-> device state movement ------------------------------------------------------ */
static void h2d_scatter(Shard &s, const double *src, int n, double *dst)
{
  if( n <= 0 ) return;
  CK(cudaMemcpyAsync(s.dstage, src + (size_t)s.e0*n, (size_t)s.B*n*sizeof(double), cudaMemcpyHostToDevice, s.stream));
  xp_scatter(s.dstage, dst, s.B, n, s.ld, s.stream, s.perm);
  CK(cudaGetLastError());
}
static void d2h_gather(Shard &s, const double *src, int n, double *dst)
{
  if( n <= 0 ) return;
  xp_gather(src, s.dstage, s.B, n, s.ld, s.stream, s.perm);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(dst + (size_t)s.e0*n, s.dstage, (size_t)s.B*n*sizeof(double), cudaMemcpyDeviceToHost, s.stream));
}

/* ---- asynchronous host <-> device movement (pinned host memory; the host buffers must stay valid and
 * unmodified until sync()).  H2D copies run on their own stream into a staging ring, the transposing scatter
 * runs on the compute stream after the copy; gathers run on the compute stream, D2H copies on a third stream:
 * transfers of step k+1 / k-1 overlap the step kernel of step k. */
static void ring_setup(Shard &s)
{
  if( s.ring_init ) return;
  CK(cudaStreamCreateWithFlags(&s.h2d_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&s.d2h_stream, cudaStreamNonBlocking));
  for(int i=0;i<Shard::NRING;i++){
    void *p = nullptr; CK(cudaMalloc(&p, s.nstage*sizeof(double))); s.allocs.push_back(p); s.ring[i] = (double*)p;
    CK(cudaEventCreateWithFlags(&s.ring_done[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&s.ring_ready[i], cudaEventDisableTiming));
  }
  s.ring_init = true;
}
static void h2d_scatter_async(Shard &s, const double *src, int n, double *dst)
{
  if( n <= 0 ) return;
  ring_setup(s);
  const int b = s.ring_next; s.ring_next = (b+1) % Shard::NRING;
  CK(cudaStreamWaitEvent(s.h2d_stream, s.ring_done[b], 0));              /* the previous user of this buffer is done */
  CK(cudaMemcpyAsync(s.ring[b], src + (size_t)s.e0*n, (size_t)s.B*n*sizeof(double), cudaMemcpyHostToDevice, s.h2d_stream));
  CK(cudaEventRecord(s.ring_ready[b], s.h2d_stream));
  CK(cudaStreamWaitEvent(s.stream, s.ring_ready[b], 0));
  xp_scatter(s.ring[b], dst, s.B, n, s.ld, s.stream, s.perm);
  CK(cudaGetLastError());
  CK(cudaEventRecord(s.ring_done[b], s.stream));
}
static void d2h_gather_async(Shard &s, const double *src, int n, double *dst)
{
  if( n <= 0 ) return;
  ring_setup(s);
  const int b = s.ring_next; s.ring_next = (b+1) % Shard::NRING;
  CK(cudaStreamWaitEvent(s.stream, s.ring_done[b], 0));
  xp_gather(src, s.ring[b], s.B, n, s.ld, s.stream, s.perm);
  CK(cudaGetLastError());
  CK(cudaEventRecord(s.ring_ready[b], s.stream));
  CK(cudaStreamWaitEvent(s.d2h_stream, s.ring_ready[b], 0));
  CK(cudaMemcpyAsync(dst + (size_t)s.e0*n, s.ring[b], (size_t)s.B*n*sizeof(double), cudaMemcpyDeviceToHost, s.d2h_stream));
  CK(cudaEventRecord(s.ring_done[b], s.d2h_stream));
}
void Engine::set_state_async(const double *q, const double *qd)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    if( q )  h2d_scatter_async(*s, q,  model_.nq, s->st.q[s->cur]);
    if( qd ) h2d_scatter_async(*s, qd, model_.nq, s->st.qd[s->cur]);
  }
  CK(cudaSetDevice(prev));
}
void Engine::set_motor_input_async(const double *u)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); h2d_scatter_async(*s, u, model_.nl, s->st.u); }
  CK(cudaSetDevice(prev));
}
void Engine::get_state_async(double *q, double *qd, double *qdd)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    if( q )   d2h_gather_async(*s, s->st.q[s->cur],  model_.nq, q);
    if( qd )  d2h_gather_async(*s, s->st.qd[s->cur], model_.nq, qd);
    if( qdd ) d2h_gather_async(*s, s->st.qdd,        model_.nq, qdd);
  }
  CK(cudaSetDevice(prev));
}
/* makes the compute stream wait for everything queued on the copy streams (so that an event recorded on the
 * compute stream afterwards covers the transfers) */
void Engine::join()
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    if( !s->ring_init ) continue;
    CK(cudaSetDevice(s->dev));
    CK(cudaEventRecord(s->ring_ready[0], s->h2d_stream)); CK(cudaStreamWaitEvent(s->stream, s->ring_ready[0], 0));
    CK(cudaEventRecord(s->ring_ready[1], s->d2h_stream)); CK(cudaStreamWaitEvent(s->stream, s->ring_ready[1], 0));
  }
  CK(cudaSetDevice(prev));
}

void Engine::set_state(const double *q, const double *qd)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    if( q )  h2d_scatter(*s, q,  model_.nq, s->st.q[s->cur]);
    if( qd ) h2d_scatter(*s, qd, model_.nq, s->st.qd[s->cur]);
  }
  /* the staging copy reads caller memory asynchronously when it is pinned: finish before returning */
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream)); }
  CK(cudaSetDevice(prev));
}
void Engine::get_state(double *q, double *qd, double *qdd)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    if( q )   d2h_gather(*s, s->st.q[s->cur],  model_.nq, q);
    if( qd )  d2h_gather(*s, s->st.qd[s->cur], model_.nq, qd);
    if( qdd ) d2h_gather(*s, s->st.qdd,        model_.nq, qdd);
  }
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream)); }
  CK(cudaSetDevice(prev));
}
void Engine::set_motor_input(const double *u)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); h2d_scatter(*s, u, model_.nl, s->st.u); }
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream)); }
  CK(cudaSetDevice(prev));
}
void Engine::set_ext_wrench(const double *w)
{
  if( model_.nfext <= 0 ) throw std::runtime_error("rokifd_b200: external wrench: no link is declared (rkFDBatchSetExtWrenchLinks)");
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); h2d_scatter(*s, w, 6*model_.nfext, s->st.fext); }
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream)); }
  CK(cudaSetDevice(prev));
}
void Engine::set_ext_wrench_device(int si, const double *w)
{
  if( model_.nfext <= 0 ) throw std::runtime_error("rokifd_b200: external wrench: no link is declared (rkFDBatchSetExtWrenchLinks)");
  if( si < 0 || si >= (int)shards_.size() ) throw std::runtime_error("rokifd_b200: external wrench: shard index out of range");
  Shard &s = *shards_[si];
  int prev = 0; CK(cudaGetDevice(&prev)); CK(cudaSetDevice(s.dev));
  /* the transposing scatter reads the caller's env-major rows through the slot permutation: no staging copy */
  xp_scatter(w, s.st.fext, s.B, 6*model_.nfext, s.ld, s.stream, s.perm);
  CK(cudaGetLastError());
  CK(cudaSetDevice(prev));
}
void Engine::set_mass_prop(const double *mp)
{
  if( model_.nmp <= 0 ) throw std::runtime_error("rokifd_b200: mass properties: no link is declared (rkFDBatchSetMassPropLinks)");
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); h2d_scatter(*s, mp, 10*model_.nmp, s->st.mp); }
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream)); }
  CK(cudaSetDevice(prev));
}
void Engine::set_mass_prop_device(int si, const double *mp)
{
  if( model_.nmp <= 0 ) throw std::runtime_error("rokifd_b200: mass properties: no link is declared (rkFDBatchSetMassPropLinks)");
  if( si < 0 || si >= (int)shards_.size() ) throw std::runtime_error("rokifd_b200: mass properties: shard index out of range");
  Shard &s = *shards_[si];
  int prev = 0; CK(cudaGetDevice(&prev)); CK(cudaSetDevice(s.dev));
  xp_scatter(mp, s.st.mp, s.B, 10*model_.nmp, s.ld, s.stream, s.perm);     /* through the slot permutation, as set_ext_wrench_device */
  CK(cudaGetLastError());
  CK(cudaSetDevice(prev));
}
/* which: 0 q, 1 q', 2 motor input; rows k0..k0+n-1 <- vals for every environment */
void Engine::fill_rows(int which, int k0, int n, const double *vals)
{
  if( n <= 0 ) return;
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    double *base = which == 0 ? s->st.q[s->cur] : ( which == 1 ? s->st.qd[s->cur] : s->st.u );
    CK(cudaMemcpyAsync(s->dstage, vals, (size_t)n*sizeof(double), cudaMemcpyHostToDevice, s->stream));
    rkfd_fill_rows_kernel<<<(s->B+255)/256, 256, 0, s->stream>>>(base + (size_t)k0*s->ld, s->ld, s->B, n, s->dstage);
    CK(cudaGetLastError());
  }
  for(Shard *s : shards_){ CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream)); }
  CK(cudaSetDevice(prev));
}

void Engine::stats(double out[8])
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(int i=0;i<8;i++) out[i] = 0.0;
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    double h[8];
    CK(cudaMemsetAsync(s->dstage, 0, 8*sizeof(double), s->stream));
    rkfd_stats_kernel<<<(s->B+255)/256, 256, 0, s->stream>>>(s->st, s->cur, model_.nq, model_.nfw, s->dstage);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h, s->dstage, sizeof h, cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    for(int i=0;i<4;i++) out[i] += h[i];
    for(int i=4;i<6;i++) if( h[i] > out[i] ) out[i] = h[i];
  }
  CK(cudaSetDevice(prev));
}

void Engine::get_pivot(int *type, double *prev_trq)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  const int nq = model_.nq;
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    if( prev_trq ) d2h_gather(*s, s->st.piv_prev, nq, prev_trq);
    CK(cudaStreamSynchronize(s->stream));
    if( type ){
      std::vector<unsigned int> bits(s->B);
      CK(cudaMemcpy(bits.data(), s->st.piv_type, s->B*sizeof(unsigned int), cudaMemcpyDeviceToHost));
      const std::vector<int> &hp = host_perm(*s);
      for(int sl=0;sl<s->B;sl++) for(int j=0;j<nq;j++) type[(size_t)(s->e0+hp[sl])*nq + j] = (bits[sl] >> j) & 1u;
    }
  }
  CK(cudaSetDevice(prev));
}
void Engine::set_pivot(const int *type, const double *prev_trq)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  const int nq = model_.nq;
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    if( prev_trq ) h2d_scatter(*s, prev_trq, nq, s->st.piv_prev);
    CK(cudaStreamSynchronize(s->stream));
    if( type ){
      std::vector<unsigned int> bits(s->B, 0u);
      const std::vector<int> &hp = host_perm(*s);
      for(int sl=0;sl<s->B;sl++) for(int j=0;j<nq;j++) if( type[(size_t)(s->e0+hp[sl])*nq + j] ) bits[sl] |= 1u << j;
      CK(cudaMemcpy(s->st.piv_type, bits.data(), s->B*sizeof(unsigned int), cudaMemcpyHostToDevice));
    }
  }
  CK(cudaSetDevice(prev));
}
void Engine::get_contact(int *active, int *type, double *ref, double *f)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  const int ns = model_.nslot;
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    if( ref ) d2h_gather(*s, s->st.cref, 3*ns, ref);
    if( f )   d2h_gather(*s, s->st.cf,   3*ns, f);
    CK(cudaStreamSynchronize(s->stream));
    if( active || type ){
      const int nfw = model_.nfw > 0 ? model_.nfw : 1;
      std::vector<unsigned long long> bits((size_t)nfw*s->ld);
      CK(cudaMemcpy(bits.data(), s->st.cflags, bits.size()*sizeof(unsigned long long), cudaMemcpyDeviceToHost));
      const std::vector<int> &hp = host_perm(*s);
      /* slot (pair, vertex) -> flag position pair.fofs + vertex */
      for(int p=0;p<model_.npair;p++){ const PairDev &pr = model_.pair[p]; const int nv = model_.cell[pr.cell].nvert;
        for(int k=0;k<nv;k++){ const int f = pr.fofs + k, sl = pr.sofs + k;
          for(int t=0;t<s->B;t++){ const unsigned long long wd = bits[(size_t)(f>>5)*s->ld + t]; const int e = hp[t];
            if( active ) active[(size_t)(s->e0+e)*ns + sl] = (int)((wd >> (2*(f&31))) & 1ull);
            if( type )   type[(size_t)(s->e0+e)*ns + sl]   = (int)((wd >> (2*(f&31)+1)) & 1ull); } } }
    }
  }
  CK(cudaSetDevice(prev));
}
void Engine::set_contact(const int *active, const int *type, const double *ref)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  const int ns = model_.nslot;
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev));
    if( ref ) h2d_scatter(*s, ref, 3*ns, s->st.cref);
    CK(cudaStreamSynchronize(s->stream));
    if( active && type ){
      const int nfw = model_.nfw > 0 ? model_.nfw : 1;
      std::vector<unsigned long long> bits((size_t)nfw*s->ld, 0ull);
      const std::vector<int> &hp = host_perm(*s);
      for(int p=0;p<model_.npair;p++){ const PairDev &pr = model_.pair[p]; const int nv = model_.cell[pr.cell].nvert;
        for(int k=0;k<nv;k++){ const int f = pr.fofs + k, sl = pr.sofs + k;
          for(int t=0;t<s->B;t++){ unsigned long long &wd = bits[(size_t)(f>>5)*s->ld + t]; const int e = hp[t];
            if( active[(size_t)(s->e0+e)*ns + sl] ) wd |= 1ull << (2*(f&31));
            if( type[(size_t)(s->e0+e)*ns + sl] )   wd |= 2ull << (2*(f&31)); } } }
      CK(cudaMemcpy(s->st.cflags, bits.data(), bits.size()*sizeof(unsigned long long), cudaMemcpyHostToDevice));
    }
  }
  CK(cudaSetDevice(prev));
}
void Engine::get_status(int *status)
{
  int prev = 0; CK(cudaGetDevice(&prev));
  for(Shard *s : shards_){
    CK(cudaSetDevice(s->dev)); CK(cudaStreamSynchronize(s->stream));
    std::vector<int> tmp(s->B); const std::vector<int> &hp = host_perm(*s);
    CK(cudaMemcpy(tmp.data(), s->st.status, s->B*sizeof(int), cudaMemcpyDeviceToHost));
    for(int sl=0;sl<s->B;sl++) status[s->e0 + hp[sl]] = tmp[sl];
  }
  CK(cudaSetDevice(prev));
}

}  // namespace rkfd
