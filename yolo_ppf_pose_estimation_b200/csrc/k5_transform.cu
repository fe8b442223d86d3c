// k5_transform.cu — K5 transform_cloud: tail of PPFRegistration::computeTransformation,
// pcl::transformPointCloud(*input_, output, results.front().pose) — xyz only, normals are not
// rotated by that overload (SURVEY.md §8 a9).
#include "ppf_common.cuh"

namespace b200ppf {

namespace {

struct Pose16 {
    float m[16];
};

__global__ void transform_cloud_kernel(const float4 *__restrict__ pos, uint32_t n, Pose16 P, float *__restrict__ out,
                                       uint32_t stride) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pos[i];
    const float *M = P.m;
    float *o = out + (size_t)i * stride;
    o[0] = ((M[0] * p.x + M[1] * p.y) + M[2] * p.z) + M[3];
    o[1] = ((M[4] * p.x + M[5] * p.y) + M[6] * p.z) + M[7];
    o[2] = ((M[8] * p.x + M[9] * p.y) + M[10] * p.z) + M[11];
}

}  // namespace

int k5_transform(b200ppf_ctx *ctx, const b200ppf_cloud *cloud, const float *pose16, float *out_host,
                 size_t out_stride_floats) {
    const size_t n = cloud->n;
    if (n == 0) return B200PPF_OK;
    if (out_stride_floats < 3) return fail_msg(ctx, B200PPF_ERR_INVALID, "transform: output stride must be >= 3 floats");
    Pose16 P;
    memcpy(P.m, pose16, sizeof(P.m));
    StreamBuf<float> d(ctx);
    PPF_CUDA(ctx, d.alloc(n * 3));
    cudaEventRecord(ctx->ev[0], ctx->stream);
    PPF_LAUNCH(ctx, transform_cloud_kernel, (unsigned)((n + 255) / 256), 256, 0, cloud->pos, (uint32_t)n, P, d, 3u);
    cudaEventRecord(ctx->ev[1], ctx->stream);
    // strided copy back: only xyz of every output element is written, the rest is the caller's
    PPF_CUDA(ctx, cudaMemcpy2DAsync(out_host, out_stride_floats * sizeof(float), d, 3 * sizeof(float), 3 * sizeof(float),
                                    n, cudaMemcpyDeviceToHost, ctx->stream));
    PPF_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->timings.transform_ms, ctx->ev[0], ctx->ev[1]);
    return B200PPF_OK;
}

}  // namespace b200ppf
