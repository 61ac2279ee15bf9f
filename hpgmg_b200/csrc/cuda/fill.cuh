/*
 * fill.cuh -- one work item of a ghost fill (see ghost.cu): either one ghost cell copied from the
 * neighbouring box on this GPU, or one boundary-condition column.  Shared by the fill kernel and the
 * persistent smoother of the small levels (smooth.cu).
 */
#ifndef HPGMG_B200_FILL_CUH
#define HPGMG_B200_FILL_CUH
#include "common.cuh"
#include "bc.cuh"

__device__ __forceinline__ void fill_items(const DLevel &L, const int id, const int t, const FillCopy *__restrict__ copies, const int ncopies,
                                           const FillBC *__restrict__ bc, const int nbc, const int version)
{
  double *v = L.base + (size_t)id * (size_t)L.volume;
  if (t < ncopies) {
    const FillCopy c = copies[t];
    v[c.dst] = v[c.src];
  } else if (t < ncopies + nbc) {
    const FillBC it = bc[t - ncopies];
    const BCNormal N = bc_normal(it.subtype, L.jStride, L.kStride);
    if (version == 4) bc_v4_column(v + it.src, v + it.dst, N);
    else              bc_v2_fill_col(v + it.src, v + it.dst, N.m, N.d[0], N.d[1], N.d[2]);
  }
}


#endif
