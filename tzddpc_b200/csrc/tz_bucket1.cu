// Kernel bucket B1 of the fused step kernel (tz_step.cuh), in its own translation unit so that the buckets compile in parallel.
#include "tz_step.cuh"

namespace tz {
template int launch_bucket<B1>(const TzProgram*, const SolverParams&, const StepArgs&, cudaStream_t);
template int launch_bucket_set<B1>(const TzProgram*, const SetEntry*, int, int64_t, const SolverParams&, const StepArgs&, cudaStream_t);
template int launch_bucket_set_run<B1>(const TzProgram*, const SetEntry*, int, int64_t, const SolverParams&, const StepArgs&, cudaStream_t);
}
