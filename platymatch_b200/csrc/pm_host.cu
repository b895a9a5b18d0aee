// pm_host.cu — host-buffer entry points (numpy callers): allocate, copy in, run, copy out, synchronise.
// These wrap the device entry points for callers that hold plain host arrays, i.e. the reference's
// own functions (platymatch/utils/utils.py:58-75, platymatch/estimate_transform/shape_context.py:144-188).
#include "pm_common.cuh"

namespace {
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes) {
        PM_CUDA_TRY(cudaMalloc(&p, bytes ? bytes : 1));
        return PM_OK;
    }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};
}  // namespace

#define PM_TRY(expr) do { int _rc = (expr); if (_rc != PM_OK) return _rc; } while (0)

extern "C" int pm_host_mean_distance(const double *pts, int n, int device, double *out_mean) {
    PM_REQUIRE(pts && out_mean, "null pointer");
    PM_REQUIRE(n >= 2, "need at least 2 points");
    PM_CUDA_TRY(cudaSetDevice(device));
    DevBuf dpts, dws, dout;
    PM_TRY(dpts.alloc((size_t)n * 3 * sizeof(double)));
    PM_TRY(dws.alloc(pm_mean_distance_workspace_bytes(n)));
    PM_TRY(dout.alloc(sizeof(double)));
    PM_CUDA_TRY(cudaMemcpy(dpts.p, pts, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice));
    PM_TRY(pm_mean_distance(dpts.as<double>(), n, dout.as<double>(), dws.p, pm_mean_distance_workspace_bytes(n), 0));
    PM_CUDA_TRY(cudaMemcpy(out_mean, dout.p, sizeof(double), cudaMemcpyDeviceToHost));
    return PM_OK;
}

extern "C" int pm_host_shape_context(const double *pts, int n, const double *centroid, double mean_dist,
                                     const double *r_edges, int n_redges, int n_variants, int device,
                                     uint32_t *counts, uint32_t *dropped, double *x0_out,
                                     unsigned long long *edge_ties_out) {
    PM_REQUIRE(pts && centroid && r_edges && counts, "null pointer");
    PM_REQUIRE(n >= 2, "need at least 2 points");
    PM_REQUIRE(n_redges >= 1 && n_redges <= 5, "n_redges must be 1..5");
    PM_CUDA_TRY(cudaSetDevice(device));
    DevBuf dpts, dstats, dsmall, dcounts, ddropped;
    const size_t cbytes = (size_t)n_variants * n * PM_NBINS * sizeof(uint32_t);
    PM_TRY(dpts.alloc((size_t)n * 3 * sizeof(double)));
    PM_TRY(dstats.alloc(PM_STATS_DOUBLES * sizeof(double)));
    PM_TRY(dsmall.alloc(16 * sizeof(double)));   // [0:3] centroid, [3] mean_dist, [4:9] r_edges, [10] ties
    PM_TRY(dcounts.alloc(cbytes));
    PM_TRY(ddropped.alloc((size_t)n_variants * n * sizeof(uint32_t)));
    double small[16] = {0};
    small[0] = centroid[0]; small[1] = centroid[1]; small[2] = centroid[2]; small[3] = mean_dist;
    for (int e = 0; e < n_redges; ++e) small[4 + e] = r_edges[e];
    PM_CUDA_TRY(cudaMemcpy(dpts.p, pts, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice));
    PM_CUDA_TRY(cudaMemcpy(dsmall.p, small, sizeof(small), cudaMemcpyHostToDevice));
    PM_TRY(pm_cloud_stats(dpts.as<double>(), n, dstats.as<double>(), 0));
    double *ds = dsmall.as<double>();
    PM_TRY(pm_shape_context_hist_rows(dpts.as<double>(), n, ds, dstats.as<double>() + 3, ds + 3, ds + 4, n_redges,
                                      n_variants, 0, n, dcounts.as<uint32_t>(), ddropped.as<uint32_t>(),
                                      reinterpret_cast<unsigned long long *>(ds + 10), 0));
    PM_CUDA_TRY(cudaMemcpy(counts, dcounts.p, cbytes, cudaMemcpyDeviceToHost));
    if (dropped)
        PM_CUDA_TRY(cudaMemcpy(dropped, ddropped.p, (size_t)n_variants * n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (x0_out) PM_CUDA_TRY(cudaMemcpy(x0_out, dstats.as<double>() + 3, 3 * sizeof(double), cudaMemcpyDeviceToHost));
    if (edge_ties_out)
        PM_CUDA_TRY(cudaMemcpy(edge_ties_out, ds + 10, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return PM_OK;
}
