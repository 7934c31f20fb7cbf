// Row-group form of the coded E-step (fcd_estep_rows.cu): host-side entry used by fcd_estep_qF_coded.
#pragma once

#include "fcd_common.cuh"

namespace fcd {

bool estep_rows_supported(int U, int64_t pitchU, int64_t pitchQ);
// S0: observed controls per edge (the masked form), or NULL
int estep_rows_launch(const double* S1, const double* S2, const double* S0, const double* P, int64_t planeStride,
                      int64_t C, int U, int64_t pitchU, const double* qR, const int32_t* nm, const uint8_t* code,
                      int64_t pitchQ, const int32_t* counts, const uint64_t* keysF, const uint64_t* keysH, const int64_t* rowoff,
                      const double* Hh, const ThetaDev& th, const LogTabWindow& tab, bool fast, double* lqF, double* qF,
                      cudaStream_t st);

}  // namespace fcd
