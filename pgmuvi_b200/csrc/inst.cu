// One translation unit per (kernel kind, padded mixture count): compiled with
//   -DPGM_INST_KIND=k -DPGM_INST_QT=q -DPGM_INST_D=d
#include "launch_impl.cuh"
namespace pgm {
template int launch_eval<PGM_INST_KIND, PGM_INST_QT, PGM_INST_D>(const EvalArgs&, cudaStream_t);
template int launch_fit<PGM_INST_KIND, PGM_INST_QT, PGM_INST_D>(const FitArgs&, cudaStream_t);
template int launch_dense<PGM_INST_KIND, PGM_INST_QT, PGM_INST_D>(const EvalArgs&, double*, cudaStream_t);
template int launch_large<PGM_INST_KIND, PGM_INST_QT, PGM_INST_D>(const LargeArgs&, int, cudaStream_t, int);
template int launch_predict<PGM_INST_KIND, PGM_INST_QT, PGM_INST_D>(const PredictArgs&, cudaStream_t);
template int launch_fisher<PGM_INST_KIND, PGM_INST_QT, PGM_INST_D>(const LargeArgs&, const FisherArgs&,
                                                                  cudaStream_t);
}  // namespace pgm
