// cell_row.cuh -- the z cell row of a marker, which decides the rank that owns it with z-slab ownership.
// The migration (migrate.cu) and the snapshot reader (output.cu) both use it, so that they always agree on
// ownership, and migrate.owner_of restates it in torch: floor((nz-1)*z/Lz) (pylamp2.py:588) with IEEE multiply
// then divide and no FMA, clamped to the cell rows [0, nz-2].
#pragma once

static __device__ __forceinline__ int row_of(double z, int nz, double Lz) {
    long long ie = (long long)floor(__ddiv_rn(__dmul_rn((double)(nz - 1), z), Lz));
    return ie < 0 ? 0 : (ie > nz - 2 ? nz - 2 : (int)ie);
}
