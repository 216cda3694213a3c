// oracle/ref_shim_metric.cpp -- TEST INFRASTRUCTURE ONLY (never linked into the product).
//
// The door of oracle/ref_shim.cpp with the reference's `manhattan_spatial_dist` field set as the caller asks
// (context.h:35; cfast_slic.pyx:186, :246 copy it onto every context).  Built by oracle/metric.mk into
// oracle/_ref/libfslic_ref_metric.so against the reference objects of oracle/_ref/libfslic_ref.so; the sources under
// /root/reference are compiled in place, never copied.
#include <cstdint>
#include "context.h"
#include "arch/x64/avx2.h"

namespace {
template <typename Base>
struct Probe : public Base {
    Probe(int H, int W, int K, const uint8_t* image, Cluster* clusters) : Base(H, W, K, image, clusters) {}
    void dump(uint16_t* precca_out) {
        if (!precca_out) return;
        for (int i = 0; i < this->H; i++)
            for (int j = 0; j < this->W; j++) precca_out[i * this->W + j] = this->assignment.get(i, j);
    }
};
// the fields SlicModel.iterate() copies in (cfast_slic.pyx:179-187)
template <typename Ctx>
void run(Ctx& ctx, uint16_t* out, int max_iter, float compactness, float min_size_factor, int stride, int convert_to_lab,
         int preemptive, float preemptive_thres, int manhattan, int num_threads, uint16_t* precca_out) {
    ctx.num_threads = num_threads;
    ctx.compactness = compactness;
    ctx.min_size_factor = min_size_factor;
    ctx.subsample_stride_config = (int16_t)stride;
    ctx.convert_to_lab = convert_to_lab != 0;
    ctx.preemptive = preemptive != 0;
    ctx.preemptive_thres = preemptive_thres;
    ctx.manhattan_spatial_dist = manhattan != 0;
    ctx.debug_mode = false;
    ctx.initialize_state();
    ctx.iterate(out, max_iter);
    ctx.dump(precca_out);
}
}  // namespace

extern "C" {

// the integer path (cfast_slic.pyx:150-197); arch: 0 = "standard", 1 = "x64/avx2"
void refm_iterate(int arch, int H, int W, int K, const uint8_t* image, Cluster* clusters, uint16_t* out, int max_iter,
                  float compactness, float min_size_factor, int stride, int convert_to_lab, int preemptive,
                  float preemptive_thres, int manhattan, int num_threads, uint16_t* precca_out) {
    if (arch == 1) {
        Probe<fslic::Context_X64_AVX2> ctx(H, W, K, image, clusters);
        run(ctx, out, max_iter, compactness, min_size_factor, stride, convert_to_lab, preemptive, preemptive_thres, manhattan,
            num_threads, precca_out);
    } else {
        Probe<fslic::Context> ctx(H, W, K, image, clusters);
        run(ctx, out, max_iter, compactness, min_size_factor, stride, convert_to_lab, preemptive, preemptive_thres, manhattan,
            num_threads, precca_out);
    }
}

// the float-distance contexts (cfast_slic.pyx:198-252): 0 = ContextRealDist, 1 = ContextRealDistL2, 2 = ContextRealDistNoQ
void refm_iterate_real(int variant, int H, int W, int K, const uint8_t* image, Cluster* clusters, uint16_t* out, int max_iter,
                       float compactness, float min_size_factor, int stride, int convert_to_lab, int manhattan,
                       int num_threads, uint16_t* precca_out) {
    if (variant == 0) {
        Probe<fslic::ContextRealDist> ctx(H, W, K, image, clusters);
        run(ctx, out, max_iter, compactness, min_size_factor, stride, convert_to_lab, 0, 0.05f, manhattan, num_threads, precca_out);
    } else if (variant == 1) {
        Probe<fslic::ContextRealDistL2> ctx(H, W, K, image, clusters);
        run(ctx, out, max_iter, compactness, min_size_factor, stride, convert_to_lab, 0, 0.05f, manhattan, num_threads, precca_out);
    } else {
        Probe<fslic::ContextRealDistNoQ> ctx(H, W, K, image, clusters);
        run(ctx, out, max_iter, compactness, min_size_factor, stride, convert_to_lab, 0, 0.05f, manhattan, num_threads, precca_out);
    }
}

}  // extern "C"
