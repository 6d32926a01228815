// fm_rows_grad.cu -- instantiations of the MODE_GRAD row kernels (one TU per mode so the families
// compile in parallel): the generic runtime-k kernel fm_rows_kernel<DEGREE, EXPLICIT, MODE, 0> for
// degree 2..6, and fm_rows_stream_kernel<.., KT> for degree 2/3 with k in {8,16,32}.
#include "fm_rows_stream.cuh"

template RowKernels row_kernels<MODE_GRAD>(int, bool, int);
