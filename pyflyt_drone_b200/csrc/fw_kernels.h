// fw_kernels.h -- internal launcher interface between fw_api.cu (C ABI, host logic) and fw_kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct FwDev;
struct FwPlanes;

#define FW_TRK_OBS 21        // the low-level tracker's observation width (task 3's observation)
#define FW_TRK_ACT 6         // and its action width

// The frozen low-level tracker of the high-level waypoint task (task 5, fw_set_tracker): device memory owned by the handle.
struct FwTrk {
    const float* params;     // policy tower of the flat (21, 6) parameter vector (include/fwppo.h layout)
    const double* stats;     // [mean 21 | var 21] frozen VecNormalize statistics, or nullptr (no normalisation)
    float clip;              // VecNormalize clip_obs
    float h_lo, h_hi, v_lo, v_hi;   // altitude / airspeed command ranges
    float* prev;             // [6][N] the tracker's previous action per env (its observation slots 12-17)
    float* obs_out;          // optional [N, 21]: raw observation of each env's last tracker decision of a step
};

// trk: the tracker of a task-5 handle (ignored by the other tasks)
cudaError_t fwk_launch_step(const FwDev& p, const FwPlanes& pl, const float* act, float* obs, float* rew, uint8_t* flg,
                            float* term_obs, bool random_act, int spl, cudaStream_t st, const FwTrk* trk = nullptr);
// zero the tracker's previous action of the envs selected by mask (device bytes, non-zero = selected)
cudaError_t fwk_launch_tracker_clear(const uint8_t* mask, float* prev, int n, cudaStream_t st);
cudaError_t fwk_graph_add_random_step(cudaGraph_t g, cudaGraphNode_t* deps, int ndeps, const FwDev& p, const FwPlanes& pl,
                                      int spl, cudaGraphNode_t* out, int pdl = 0);
bool fwk_step_supports_pdl(const FwDev& p);
cudaError_t fwk_launch_reset(const FwDev& p, const FwPlanes& pl, const uint8_t* mask, float* obs, bool emit_only,
                             cudaStream_t st);
cudaError_t fwk_launch_refill(const FwDev& p, const FwPlanes& pl, const int2* list, int* count, int* blocks_done, int cap,
                              int whole_batch, cudaStream_t st);
cudaError_t fwk_graph_add_refill(cudaGraph_t g, cudaGraphNode_t* deps, int ndeps, const FwDev& p, const FwPlanes& pl,
                                 const int2* list, int* count, int* blocks_done, int cap, cudaGraphNode_t* out);
cudaError_t fwk_launch_warm(const FwDev& p, const FwPlanes& pl, float* out, cudaStream_t st);
cudaError_t fwk_fma_peak(int sm_count, int iters, float* scratch, double* flops_per_launch, cudaStream_t st);
// debug frame of one env (fw_render.cu): rgba [H,W,4], seg [H,W], depth [H,W] device buffers, any may be null
cudaError_t fwk_render(const FwDev& p, const FwPlanes& pl, int env, int W, int H, uint8_t* rgba, int32_t* seg, float* depth,
                       cudaStream_t st);
