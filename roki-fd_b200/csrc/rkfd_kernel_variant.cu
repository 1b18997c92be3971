/* rkfd_kernel_variant.cu - one (RKFD_BLOCK, RKFD_GSCR, RKFD_RIGID, RKFD_SPEC, RKFD_MINB) instantiation of rkfd_step_kernel. */
#include "rkfd_kernel.cuh"

#ifndef RKFD_BLOCK
#error "compile with -DRKFD_BLOCK=.. -DRKFD_GSCR=.. -DRKFD_RIGID=.. -DRKFD_SPEC=.."
#endif
#ifndef RKFD_MINB
#define RKFD_MINB 1
#endif
#define RKFD_CAT_(a,b,c,d,e,f) a##b##_##c##_##d##_##e##_##f
#define RKFD_CAT(a,b,c,d,e,f) RKFD_CAT_(a,b,c,d,e,f)

namespace rkfd {

static void launch(const StateDev &st, int cur, int mode, int nsteps, int grid, size_t smem, cudaStream_t stream)
{
  rkfd_step_kernel<RKFD_BLOCK, RKFD_GSCR != 0, RKFD_RIGID != 0, RKFD_SPEC, RKFD_MINB><<<grid, RKFD_BLOCK, smem, stream>>>(st, cur, mode, nsteps, st.fext, st.mp);
}
static int blocks_per_sm(size_t smem)
{
  auto k = rkfd_step_kernel<RKFD_BLOCK, RKFD_GSCR != 0, RKFD_RIGID != 0, RKFD_SPEC, RKFD_MINB>;
  if( cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ){ cudaGetLastError(); return -1; }
  int nb = 0;
  if( cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k, RKFD_BLOCK, smem) != cudaSuccess ){ cudaGetLastError(); return -1; }
  if( SpecOf<RKFD_SPEC>::type::TM ){
    /* the occupancy query answers 1 for kernels that allocate tensor memory; the hardware co-schedules CTAs as
     * long as registers, shared memory and the 512 tensor-memory columns allow (tools/micro/tmem_scratch_test.cu) */
    cudaFuncAttributes a; int dev = 0, regs_sm = 0, smem_sm = 0, resv = 0;
    if( cudaFuncGetAttributes(&a, k) != cudaSuccess || cudaGetDevice(&dev) != cudaSuccess ){ cudaGetLastError(); return nb; }
    cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&resv, cudaDevAttrReservedSharedMemoryPerBlock, dev);
    const int regs_warp = ((a.numRegs*32 + 255)/256)*256, warps = RKFD_BLOCK/32;
    int n = regs_sm/(regs_warp*warps);
    const int by_smem = (int)((size_t)smem_sm/(smem + a.sharedSizeBytes + (size_t)resv));
    const int by_tmem = 512/(SpecOf<RKFD_SPEC>::type::TCOLS*((RKFD_BLOCK + 127)/128)), by_thr = 2048/RKFD_BLOCK;
    if( by_smem < n ) n = by_smem; if( by_tmem < n ) n = by_tmem; if( by_thr < n ) n = by_thr;
    if( n > nb ) nb = n;
  }
  return nb;
}
static int upload(const ModelDev *m, cudaStream_t stream)
{
  return (int)cudaMemcpyToSymbolAsync(c_model, m, sizeof(ModelDev), 0, cudaMemcpyHostToDevice, stream);
}
extern const KernelVariant RKFD_CAT(rkfd_variant_, RKFD_BLOCK, RKFD_GSCR, RKFD_RIGID, RKFD_SPEC, RKFD_MINB) = { RKFD_BLOCK, RKFD_GSCR != 0, RKFD_RIGID != 0, RKFD_SPEC, RKFD_MINB, launch, blocks_per_sm, upload };

}  // namespace rkfd
