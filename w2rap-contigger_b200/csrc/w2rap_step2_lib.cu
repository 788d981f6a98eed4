// w2rap_step2_lib.cu — single translation unit of the CUDA library (kernels live in headers).
#include "pipeline.cu"
#include "coverage.cu"
#include "synth.cu"
