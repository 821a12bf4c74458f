// car_waypoint_step_kernel for envs with hazards, in a translation unit of its own: compiled next to the
// instantiation without hazards, it changes how nvcc allocates that kernel's registers.
#include "waypoints.cuh"

namespace mr {

int car_waypoint_step_hazards(mr_env* env, const float2* act, float* obs, const WaypointStep& w, cudaStream_t s) {
    static OncePerDevice once;
    if (once.first())
        MR_CUDA(cudaFuncSetAttribute(car_waypoint_step_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)CAR_SMEM));
    car_waypoint_step_kernel<true><<<ceil_div(env->n, CAR_THREADS), CAR_THREADS, CAR_SMEM, s>>>(env->car, env->carK,
                                                                                                env->cfg, act, obs, w);
    MR_CHECK_LAUNCH();
    return MR_OK;
}

}  // namespace mr
