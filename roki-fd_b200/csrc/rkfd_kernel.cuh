/* rkfd_kernel.cuh - the fused step kernel template and its device context.  Each (BLOCK, GSCR, RIGID, SPEC)
 * variant is compiled in its own translation unit (rkfd_kernel_variant.cu with -D flags) so that the
 * variants build in parallel and the penalty-only kernels carry no rigid-solver code. */
#ifndef RKFD_KERNEL_CUH
#define RKFD_KERNEL_CUH

#include <cuda_runtime.h>
#include <cstdio>

#include "rkfd_core.cuh"

namespace rkfd {

/* per-variant copy of the model table (each translation unit is its own module with its own constant bank) */
static __constant__ ModelDev c_model;

extern __shared__ double rkfd_smem[];

/* tensor memory as per-thread scratch: one TMEM lane per thread (warp w of the CTA owns lanes 32*(w%4)..+31),
 * element k of the thread = 32-bit columns 2k, 2k+1.  tcgen05.ld/st are warp-collective (.sync.aligned): every
 * T-space access sits in warp-uniform code. */
/* columns per warpgroup: Spec::TCOLS (128 = 64 doubles per thread for the arm specialisations, 256 for the generic kernel) */

template <int BLOCK, bool GSCR, bool RIGID_, bool TM>
struct DevCtx {
  /* (the tensor-memory columns per warpgroup only enter the kernel prologue: tbase) */
  static constexpr bool RIGID = RIGID_;
  StateDev st; int e, cur, tid;     /* e / tid: the SELECTED environment / scratch column (own, except in cooperative sections) */
  int e0, tid0, wsd;
  unsigned tbase;                   /* tensor-memory address of element 0 of this thread's lane (TM variants) */
  __device__ __forceinline__ double TL(int k){
    if( !TM ) return S(k);
    unsigned lo, hi;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(tbase + 2u*(unsigned)k));
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(lo), "+r"(hi) :: "memory");
    return __hiloint2double((int)hi, (int)lo);
  }
  /* elements k, k+1 with one instruction */
  __device__ __forceinline__ void TL2(int k, double &a, double &b){
    if( !TM ){ a = S(k); b = S(k+1); return; }
    unsigned r0, r1, r2, r3;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(tbase + 2u*(unsigned)k));
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r0), "+r"(r1), "+r"(r2), "+r"(r3) :: "memory");
    a = __hiloint2double((int)r1, (int)r0); b = __hiloint2double((int)r3, (int)r2);
  }
  __device__ __forceinline__ void TS(int k, double v){
    if( !TM ){ S(k) = v; return; }
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" :: "r"(tbase + 2u*(unsigned)k), "r"(__double2loint(v)), "r"(__double2hiint(v)) : "memory");
  }
  __device__ __forceinline__ void tfence(){
    if( TM ){
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
  }
  /* scratch element k of this thread: shared-memory column [k*BLOCK + tid] (LDS/STS, conflict-free) */
#ifdef RKFD_BOUNDS      /* debug build (compute-sanitizer is not available on the pool): the first out-of-range index is recorded
                         * in the environment's status word (bit 30 set, bits 24-27 which accessor, bits 0-23 the index) */
  int oob, bnd_ns, bnd_w1;
  __device__ __forceinline__ int chk(int k, int n, int which){ if( (unsigned)k >= (unsigned)n ){ if( !oob ) oob = (1 << 30) | (which << 24) | (k & 0xffffff); return 0; } return k; }
#endif
  __device__ __forceinline__ double &S(int k){
#ifdef RKFD_BOUNDS
    k = chk(k, bnd_ns, 1);
#endif
    if( GSCR ) return st.scratch[(size_t)k*st.ld + e];
    return rkfd_smem[k*BLOCK + tid];
  }
  /* warp-cooperative sections: all 32 lanes work on the environment of lane `src` */
  __device__ __forceinline__ int lanes() const { return 32; }
  __device__ __forceinline__ int lane() const { return tid0 & 31; }
  __device__ __forceinline__ unsigned ballot(bool p) const { return __ballot_sync(0xffffffffu, p); }
  __device__ __forceinline__ bool any(bool p) const { return __any_sync(0xffffffffu, p); }
  __device__ __forceinline__ unsigned long long bcast(unsigned long long x, int src) const { return __shfl_sync(0xffffffffu, x, src); }
  __device__ __forceinline__ double allsum(double x) const {
#pragma unroll
    for(int o=16;o>0;o>>=1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x; }
  __device__ __forceinline__ void select(int src){ tid = (tid0 & ~31) | src; e = (e0 & ~31) | src; }
  __device__ __forceinline__ void unselect(){ tid = tid0; e = e0; }
  __device__ __forceinline__ void gsync() const { __syncwarp(); }
  /* Reconvergence that the compiler cannot drop: at a point it takes for convergent (the head of a loop with a warp-uniform
   * trip count) it deletes __syncwarp() and issues the vote for the lanes that happen to be there - lanes that skipped a
   * divergent body with calls in it then run ahead, through the block barriers as well (an aligned barrier counts a part of
   * a warp as the warp), and overwrite the uniform registers of the lanes still in the body (seen on the B200 as "warp
   * out-of-range address").  With a mask the compiler cannot evaluate (all ones for any valid launch) the warp barrier stays. */
  __device__ __forceinline__ unsigned hmask() const { return ~(unsigned)(st.B >> 31); }
  __device__ __forceinline__ void hsync() const { __syncwarp(hmask()); }
  __device__ __forceinline__ bool hany(bool p) const { const unsigned fm = hmask(); __syncwarp(fm); return __any_sync(fm, p); }
  __device__ __forceinline__ bool block_or(bool p) const { return __syncthreads_or(p) != 0; }     /* block-uniform call sites only */
#ifndef RKFD_SYNC_LEVEL
#define RKFD_SYNC_LEVEL 2
#endif
  /* level 1: once per evaluation, 2: per pass, 3: per link iteration */
  __device__ __forceinline__ void phase_sync(int level) const { if( level <= RKFD_SYNC_LEVEL ) __syncthreads(); }
  __device__ __forceinline__ double &W(int i){ return st.ws[(size_t)(e0 >> 5)*wsd + i]; }
  __device__ __forceinline__ double &W1(int i){
#ifdef RKFD_BOUNDS
    i = chk(i, bnd_w1, 2);
#endif
    return st.ws1[(size_t)i*st.ld + e]; }     /* element i of the selected environment */
  /* per-env state in HBM: element k of the selected environment (global address space asserted: LDG/STG, not generic) */
  /* the element index k*ld + e in 32 bits (one IMAD + one IMAD.WIDE per access instead of a 64-bit multiply-add chain: the
   * address arithmetic of these accesses was 5 % of the executed instructions of the C3 step); the engine refuses batches whose
   * largest row index times ld does not fit (Engine::Engine) */
  __device__ __forceinline__ double gld(const double *p, int k) const { const double *a = p + ((unsigned)k*(unsigned)st.ld + (unsigned)e); __builtin_assume(__isGlobal(a)); return *a; }
  __device__ __forceinline__ void gst(double *p, int k, double v){ double *a = p + ((unsigned)k*(unsigned)st.ld + (unsigned)e); __builtin_assume(__isGlobal(a)); *a = v; }
};

/* mode 0: nsteps x rkFDUpdate; 1: one non-committing evaluation; 2: one committing evaluation */
/* MINB (minimum resident blocks per SM, i.e. the register cap) is a template parameter so that every compiled
 * variant has its own kernel symbol: two translation units instantiating the same template arguments with
 * different launch bounds would collide at link time and launch each other's module (and constant bank). */
template <int BLOCK, bool GSCR, bool RIGID, int SPEC, int MINB>
__global__ void __launch_bounds__(BLOCK, MINB) rkfd_step_kernel(StateDevHead sh, int cur, int mode, int nsteps, double *fext, double *mp)
{
  StateDev st; static_cast<StateDevHead &>(st) = sh; st.fext = fext; st.mp = mp;
  using Spec = typename SpecOf<SPEC>::type;
  constexpr bool TM = Spec::TM != 0;
  int e_ = blockIdx.x*BLOCK + threadIdx.x;
  asm volatile("" : "+r"(e_));        /* opaque: kept in a register instead of being recomputed from the special registers at every use */
  const int e = e_;
  /* the engine pads the environment count to whole blocks (ld): no thread exits early, which the block barriers
   * and the tensor-memory allocation below rely on; the padding environments hold a valid zero state */
  int tid_ = threadIdx.x;
  asm volatile("" : "+r"(tid_));      /* opaque, like e: the scratch-column index is not re-read from the special register at every access */
  DevCtx<BLOCK,GSCR,RIGID,TM> ctx; ctx.st = st; ctx.e = ctx.e0 = e; ctx.cur = cur; ctx.tid = ctx.tid0 = tid_; ctx.wsd = c_model.ws_doubles;
  ctx.tbase = 0;
#ifdef RKFD_BOUNDS
  ctx.oob = 0; ctx.bnd_ns = c_model.nscratch; ctx.bnd_w1 = c_model.ws1_doubles > 0 ? c_model.ws1_doubles : 1;
#endif
  constexpr unsigned TCOLS = Spec::TCOLS*((BLOCK + 127)/128);
  __shared__ unsigned tmem_addr;
  if( TM ){
    static_assert(!TM || ((TCOLS & (TCOLS-1)) == 0 && TCOLS >= 32 && TCOLS <= 512), "tensor-memory columns: power of two in [32, 512]");
    static_assert(!TM || 2*Spec::NTSPACE <= Spec::TCOLS, "T space does not fit the tensor-memory lane");
    if( threadIdx.x < 32 ){
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"((unsigned)__cvta_generic_to_shared(&tmem_addr)), "r"(TCOLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned warp = threadIdx.x >> 5;
    ctx.tbase = tmem_addr + (((warp & 3u)*32u) << 16) + (warp >> 2)*Spec::TCOLS;
  }
  Core<DevCtx<BLOCK,GSCR,RIGID,TM>, Spec> core(ctx);
  core.run(c_model, mode, nsteps);
#ifdef RKFD_BOUNDS
  if( ctx.oob ) st.status[ctx.e0] = ctx.oob;
#endif
  if( TM ){
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if( threadIdx.x < 32 )
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_addr), "r"(TCOLS) : "memory");
  }
}


/* one compiled variant: launch + occupancy query */
struct KernelVariant {
  int block; bool gscr, rigid; int spec;     /* spec: model specialisation id (rkfd_core.cuh), 0 = generic */
  int minb;                                  /* __launch_bounds__ minimum blocks per SM the variant was compiled for */
  void (*launch)(const StateDev &st, int cur, int mode, int nsteps, int grid, size_t smem, cudaStream_t stream);
  int (*blocks_per_sm)(size_t smem);      /* sets the dynamic shared memory attribute; <0 on error */
  int (*upload)(const ModelDev *m, cudaStream_t stream);   /* model table -> this variant's constant bank */
};

}  // namespace rkfd
#endif
