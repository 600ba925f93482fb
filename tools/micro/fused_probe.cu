// fused_probe.cu -- per-phase clock64() breakdown of k_step_fused on one 128 x 128 simulation per SM.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -DSMK_FUSED_TIMING -I smokephysai_b200/csrc -o build/fused_probe tools/micro/fused_probe.cu
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cmath>
namespace smk { int fail(int c, const char*, ...) { return c; } int check_launch(const char*) { return 0; } }
#include "fused.cu"
namespace smk { void prof_mark(int, cudaStream_t, bool) {} }
using namespace smk;

int main(int argc, char** argv)
{
    const int K = argc > 1 ? atoi(argv[1]) : 40, nsteps = argc > 2 ? atoi(argv[2]) : 8, B = 148;
    const size_t nu = 129 * 128, nv = 128 * 132, nc = 128 * 128;
    std::vector<float> hd(B * nc, 0.f);
    for (int b = 0; b < B; ++b)
        for (int e = 0; e < 2; ++e) {
            const int cx = 30 + (b * 7 + e * 41) % 70, cy = 30 + (b * 13 + e * 29) % 70;
            for (int i = 0; i < 128; ++i)
                for (int j = 0; j < 128; ++j) {
                    const float d2 = (float)((i - cy) * (i - cy) + (j - cx) * (j - cx));
                    if (d2 <= 64.f) hd[b * nc + i * 128 + j] += 1.5f * expf(-d2 / (2.f * (8.f / 3.f) * (8.f / 3.f)));
                }
        }
    float *u, *v, *d, *p, *fr; long long* ticks;
    cudaMalloc(&u, B * nu * 4); cudaMalloc(&v, B * nv * 4); cudaMalloc(&d, B * nc * 4); cudaMalloc(&p, B * nc * 4);
    cudaMalloc(&fr, (size_t)B * nsteps * nc * 4); cudaMalloc(&ticks, 8 * 8);
    cudaMemset(u, 0, B * nu * 4); cudaMemset(v, 0, B * nv * 4); cudaMemset(p, 0, B * nc * 4);
    cudaMemcpy(d, hd.data(), B * nc * 4, cudaMemcpyHostToDevice);
    cudaFuncSetAttribute(k_step_fused<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FZ_SMEM);
    FusedArgs a;
    a.U = u; a.V = v; a.D = d; a.P = p; a.frames = fr; a.fmul = nullptr;
    a.h = 128; a.w = 128; a.pu = 128; a.pv = 132; a.pc = 128; a.su_ = nu; a.sv_ = nv; a.sc_ = nc;
    a.frame_step_stride = nc; a.frame_batch_stride = (long long)nsteps * nc;
    a.dt = 0.01f; a.c_uv = (float)(0.01 * 0.001); a.c_d = (float)(0.01 * (0.001 * 0.1)); a.decay = 0.995f; a.K = K; a.nsteps = nsteps;
    a.ticks = ticks;
    for (int rep = 0; rep < 3; ++rep) {
        cudaMemset(ticks, 0, 64);
        k_step_fused<true, false><<<B, FZ_THREADS, FZ_SMEM>>>(a);
        cudaDeviceSynchronize();
    }
    long long t[8];
    cudaMemcpy(t, ticks, 64, cudaMemcpyDeviceToHost);
    const char* names[8] = {"load + first buoyancy", "diffusion x3", "divergence", "jacobi", "gradient subtract", "advection x3", "frame + buoyancy", "store"};
    long long per_step = 0;
    for (int k = 1; k <= 6; ++k) per_step += t[k];
    printf("K=%d, %d steps per launch, %s\n", K, nsteps, cudaGetErrorString(cudaGetLastError()));
    for (int k = 0; k < 8; ++k) {
        const bool once = (k == 0 || k == 7);
        printf("  %-24s %9.0f cycles %s  %5.1f %% of a step\n", names[k], once ? (double)t[k] : (double)t[k] / nsteps, once ? "per launch" : "per step  ",
               100.0 * (once ? (double)t[k] : (double)t[k] / nsteps) / ((double)per_step / nsteps));
    }
    printf("  step total %.0f cycles\n", (double)per_step / nsteps);
    return 0;
}
