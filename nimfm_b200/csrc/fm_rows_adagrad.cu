// fm_rows_adagrad.cu -- instantiations of the MODE_ADAGRAD row kernels: the generic runtime-k kernel
// for degree 2..6 and the register-streaming kernel for degree 2/3 with k in {8,16,32}.
#include "fm_rows_stream.cuh"

template RowKernels row_kernels<MODE_ADAGRAD>(int, bool, int);
