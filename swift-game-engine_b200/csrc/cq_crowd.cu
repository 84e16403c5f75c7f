// cq_crowd.cu — resident crowd (include/cq.h): character records stay in HBM between steps; a step moves velocities in
// and poses out (24 + 56 bytes per character) instead of the full 168-byte record each way.
//
// Why: cq_move_and_slide_batch is PCIe bound — 2 x 176 MB per step for 1,048,576 characters is >= 3.9 ms on a link that
// gives ~45 GB/s each way, against a 2.5 ms kernel.  The records are private to KinematicMoveStopSystem in the reference
// too; what crosses that system's boundary every frame is PhysicsBodyComponent.linearVelocity (written by GravitySystem /
// PhysicsIntentSystem) and the pose it leaves behind.
//
// The step is the same three-stage pipeline as the host-pointer batch calls (cq_api.cu: run_batch): a dedicated H2D stream,
// two alternating compute streams, a dedicated D2H stream, events between them.  Per chunk the compute stream runs
//   k_crowd_set_velocity  ->  k_move_and_slide (launch_move_and_slide on the chunk's slice of the resident records)
//   ->  k_crowd_get_pose.
#include <chrono>

#include "cq_internal.h"

struct cq_crowd {
    cq_world *w = nullptr;
    int n = 0;
    cq_character_state *dStates = nullptr;
    double *dVelIn = nullptr;      // n * 3
    cq_crowd_pose *dPose = nullptr; // n
    float hint = 0.0f;              // wall / PCIe ratio of the previous step (chunking heuristic, pipeline_chunks)
};

namespace cq {

__global__ void k_crowd_set_velocity(cq_character_state *__restrict__ states, const double *__restrict__ vel, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    states[i].velocity[0] = vel[3 * (size_t)i];
    states[i].velocity[1] = vel[3 * (size_t)i + 1];
    states[i].velocity[2] = vel[3 * (size_t)i + 2];
}

__global__ void k_crowd_get_pose(const cq_character_state *__restrict__ states, cq_crowd_pose *__restrict__ pose, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const cq_character_state &s = states[i];
    cq_crowd_pose p;
    p.position[0] = s.position[0], p.position[1] = s.position[1], p.position[2] = s.position[2];
    p.velocity[0] = s.velocity[0], p.velocity[1] = s.velocity[1], p.velocity[2] = s.velocity[2];
    p.ground_triangle_index = s.ground_triangle_index;
    p.grounded = s.grounded, p.grounded_near = s.grounded_near, p.ground_sliding = s.ground_sliding, p._pad = 0;
    pose[i] = p;
}

} // namespace cq

using namespace cq;

static_assert(sizeof(cq_crowd_pose) == 56, "cq_crowd_pose is 56 bytes");

extern "C" {

int cq_crowd_create(cq_world *w, const cq_character_state *initial, int32_t n, cq_crowd **out) {
    if (!w || !out || n < 0 || (n > 0 && !initial)) {
        set_error("cq_crowd_create: invalid arguments");
        return CQ_ERR_INVALID;
    }
    *out = nullptr;
    CQ_CUDA(cudaSetDevice(w->device));
    cq_crowd *c = new cq_crowd();
    c->w = w;
    c->n = n;
    const size_t cap = (size_t)std::max(n, 1);
    int rc = check_cuda(cudaMalloc((void **)&c->dStates, cap * sizeof(cq_character_state)), "crowd records");
    if (rc == CQ_OK) rc = check_cuda(cudaMalloc((void **)&c->dVelIn, cap * 3 * sizeof(double)), "crowd velocities");
    if (rc == CQ_OK) rc = check_cuda(cudaMalloc((void **)&c->dPose, cap * sizeof(cq_crowd_pose)), "crowd poses");
    if (rc == CQ_OK && n > 0)
        rc = check_cuda(cudaMemcpy(c->dStates, initial, (size_t)n * sizeof(cq_character_state), cudaMemcpyHostToDevice), "crowd upload");
    if (rc != CQ_OK) {
        cq_crowd_destroy(c);
        return rc;
    }
    *out = c;
    return CQ_OK;
}

void cq_crowd_destroy(cq_crowd *c) {
    if (!c) return;
    cudaSetDevice(c->w->device);
    cudaDeviceSynchronize(); // steps may still be in flight on the world's streams
    cudaFree(c->dStates), cudaFree(c->dVelIn), cudaFree(c->dPose);
    delete c;
}

int32_t cq_crowd_size(const cq_crowd *c) { return c ? c->n : 0; }

cq_character_state *cq_crowd_device_states(cq_crowd *c) { return c ? c->dStates : nullptr; }

int cq_crowd_read(cq_crowd *c, cq_character_state *out) {
    if (!c || (c->n > 0 && !out)) return CQ_ERR_INVALID;
    CQ_CUDA(cudaSetDevice(c->w->device));
    CQ_CUDA(cudaDeviceSynchronize());
    if (c->n) CQ_CUDA(cudaMemcpy(out, c->dStates, (size_t)c->n * sizeof(cq_character_state), cudaMemcpyDeviceToHost));
    return CQ_OK;
}

int cq_crowd_write(cq_crowd *c, const cq_character_state *in) {
    if (!c || (c->n > 0 && !in)) return CQ_ERR_INVALID;
    CQ_CUDA(cudaSetDevice(c->w->device));
    CQ_CUDA(cudaDeviceSynchronize());
    if (c->n) CQ_CUDA(cudaMemcpy(c->dStates, in, (size_t)c->n * sizeof(cq_character_state), cudaMemcpyHostToDevice));
    return CQ_OK;
}

int cq_crowd_step(cq_crowd *c, const double *velocity_in_xyz, const cq_controller_params *params, float dt, const float gravity[3],
                  uint32_t flags, const cq_platform *platforms, int32_t n_platforms, cq_crowd_pose *pose_out) {
    if (!c || !params || !gravity || n_platforms < 0 || (n_platforms > 0 && !platforms)) return CQ_ERR_INVALID;
    cq_world *w = c->w;
    const int n = c->n;
    if (n == 0) return CQ_OK;
    CQ_CUDA(cudaSetDevice(w->device));
    CQ_NO_CAPTURE(w->stream, "cq_crowd_step");
    CQ_CUDA(cudaStreamSynchronize(w->stream));
    static const float HINT = [] { // wall / PCIe-time ratio above which the step counts as compute bound (CQ_CROWD_HINT overrides)
        const char *e = getenv("CQ_CROWD_HINT");
        const float v = e ? (float)atof(e) : 0.0f;
        return v > 0.0f ? v : 3.0f;
    }();
    // CQ_MAS_AGENTS: the characters interact, all velocities must be in place before the kernel starts
    const int nChunks = pipeline_chunks(n, c->hint, HINT, (flags & CQ_MAS_AGENTS) != 0);
    const auto t0 = std::chrono::steady_clock::now();
    const int chunk = (n + nChunks - 1) / nChunks;
    int k = 0;
    for (int lo = 0; lo < n; lo += chunk, k++) {
        const int cnt = std::min(chunk, n - lo);
        cudaStream_t cs = w->copyStream[k & 1];
        cq_character_state *dS = c->dStates + lo;
        if (velocity_in_xyz) {
            CQ_CUDA(cudaMemcpyAsync(c->dVelIn + 3 * (size_t)lo, velocity_in_xyz + 3 * (size_t)lo, sizeof(double) * 3 * (size_t)cnt,
                                    cudaMemcpyHostToDevice, w->h2dStream));
            CQ_CUDA(cudaEventRecord(w->evIn[k], w->h2dStream));
            CQ_CUDA(cudaStreamWaitEvent(cs, w->evIn[k], 0));
            k_crowd_set_velocity<<<(cnt + 255) / 256, 256, 0, cs>>>(dS, c->dVelIn + 3 * (size_t)lo, cnt);
            w->launches++;
        }
        CQ_TRY(launch_move_and_slide(w, dS, cnt, *params, dt, gravity, flags, platforms, nullptr, n_platforms, cs));
        if (pose_out) {
            k_crowd_get_pose<<<(cnt + 255) / 256, 256, 0, cs>>>(dS, c->dPose + lo, cnt);
            w->launches++;
            CQ_CUDA(cudaGetLastError());
            CQ_CUDA(cudaEventRecord(w->evDone[k], cs));
            CQ_CUDA(cudaStreamWaitEvent(w->d2hStream, w->evDone[k], 0));
            CQ_CUDA(cudaMemcpyAsync(pose_out + lo, c->dPose + lo, sizeof(cq_crowd_pose) * (size_t)cnt, cudaMemcpyDeviceToHost,
                                    w->d2hStream));
        }
    }
    // the call is synchronous: everything it enqueued has finished when it returns
    CQ_CUDA(cudaStreamSynchronize(w->copyStream[0]));
    CQ_CUDA(cudaStreamSynchronize(w->copyStream[1]));
    CQ_CUDA(cudaStreamSynchronize(w->d2hStream));
    const double wallMs = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    const double pcieMs = (double)n * 56.0 / 50.0e6;
    c->hint = (float)(wallMs / std::max(pcieMs, 1e-3));
    return CQ_OK;
}

} // extern "C"
