// harness.cu -- runs block_seqsum_exact_v2 (csrc/seqsum2.cuh) against the literal float loop on the
// adversarial generators of proto.c and times it.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -fmad=false -I gpullama3.java_b200/csrc -o /tmp/seqsum2_harness tools/seqsum2/harness.cu
#include "seqsum2.cuh"
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

__global__ void __launch_bounds__(SEQSUM2_THREADS, 1) k_v2(const float *t, int n, float *out, int *info) {
    extern __shared__ __align__(16) unsigned char sm2[];
    const int E = (n + SEQSUM2_THREADS - 1) / SEQSUM2_THREADS, np = SEQSUM2_THREADS * E;
    float *sq = reinterpret_cast<float *>(sm2);
    SeqSum2Scratch sc = seqsum2_carve(sm2 + (size_t)np * 4);
    for (int i = threadIdx.x; i < np; i += SEQSUM2_THREADS) sq[i] = i < n ? t[i] : 0.0f;
    __syncthreads();
    const float s = block_seqsum_exact_v2(sq, n, sc);
    if (threadIdx.x == 0) { out[0] = s; info[0] = sc.info[0]; info[1] = sc.info[1]; }
}
// the 256-thread form the persistent decode kernel uses (every CTA sums redundantly with its 8 consumer warps)
__global__ void __launch_bounds__(256, 1) k_v2_256(const float *t, int n, float *out, int *info) {
    extern __shared__ __align__(16) unsigned char sm3[];
    const int E = (n + 255) / 256, np = 256 * E;
    float *sq = reinterpret_cast<float *>(sm3);
    SeqSum2Scratch sc = seqsum2_carve(sm3 + (size_t)np * 4);
    for (int i = threadIdx.x; i < np; i += 256) sq[i] = i < n ? t[i] : 0.0f;
    __syncthreads();
    const float s = block_seqsum_exact_v2_t<256>(sq, n, sc, (int)threadIdx.x, SeqSum2BlockSync());
    if (threadIdx.x == 0) { out[0] = s; info[0] = sc.info[0]; info[1] = sc.info[1]; }
}

static unsigned long long rng = 88172645463325252ull;
static unsigned xr() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return (unsigned)(rng >> 16); }
static float urand() { return (xr() & 0xffffff) / 16777216.0f; }
static float nrand() { float u = urand() + 1e-7f, v = urand(); return sqrtf(-2.f * logf(u)) * cosf(6.2831853f * v); }

int main(int argc, char **argv) {
    const int n = argc > 1 ? atoi(argv[1]) : 4096, cases = argc > 2 ? atoi(argv[2]) : 2000;
    std::vector<float> t(n);
    float *dt, *dout;
    int *dinfo;
    cudaMalloc(&dt, n * 4); cudaMalloc(&dout, 16); cudaMalloc(&dinfo, 16);
    const int E = (n + SEQSUM2_THREADS - 1) / SEQSUM2_THREADS;
    const size_t smem2 = (size_t)SEQSUM2_THREADS * E * 4 + seqsum2_scratch_bytes();
    cudaFuncSetAttribute(k_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
    const size_t smem3 = (size_t)256 * ((n + 255) / 256) * 4 + seqsum2_scratch_bytes();
    cudaFuncSetAttribute(k_v2_256, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3);
    long bad = 0, items = 0, fb = 0;
    for (int c = 0; c < cases; c++) {
        const int kind = c % 10;
        for (int i = 0; i < n; i++) {
            float x;
            switch (kind) {
            case 0: x = nrand(); break;
            case 1: x = nrand() * 0.02f; break;
            case 2: x = nrand() * (i % 97 == 0 ? 30.f : 1.f); break;
            case 3: x = ldexpf(1.0f, (int)(xr() % 12) - 6); break;
            case 4: x = (float)(xr() % 8) * 0.25f; break;
            case 5: x = (i < n / 2) ? 1e-3f * urand() : 50.f * urand(); break;
            case 6: x = (xr() % 50 == 0) ? nrand() * 100.f : 0.f; break;
            case 7: x = sqrtf(ldexpf(1.0f + urand() * 1e-3f, (int)(xr() % 3))); break;
            case 8: x = nrand() * expf(nrand()); break;
            default: x = (c & 16) ? 1.0f : 0.5f; break;
            }
            t[i] = x * x;
        }
        volatile float s = 0.f;
        for (int i = 0; i < n; i++) s = s + t[i];
        cudaMemcpy(dt, t.data(), n * 4, cudaMemcpyHostToDevice);
        k_v2<<<1, SEQSUM2_THREADS, smem2>>>(dt, n, dout, dinfo);
        float got;
        int info[2];
        cudaMemcpy(&got, dout, 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(info, dinfo, 8, cudaMemcpyDeviceToHost);
        float ref = s;
        if (memcmp(&got, &ref, 4)) { if (bad < 5) printf("MISMATCH case %d kind %d: gpu %.9g literal %.9g\n", c, kind, got, ref); bad++; }
        k_v2_256<<<1, 256, smem3>>>(dt, n, dout, dinfo);
        cudaMemcpy(&got, dout, 4, cudaMemcpyDeviceToHost);
        if (memcmp(&got, &ref, 4)) { if (bad < 5) printf("MISMATCH (256 threads) case %d kind %d: gpu %.9g literal %.9g\n", c, kind, got, ref); bad++; }
        items += info[0]; fb += info[1];
    }
    printf("n=%d cases=%d mismatches=%ld items/case=%.1f fallbacks/case=%.3f (%s)\n", n, cases, bad, (double)items / cases, (double)fb / cases, cudaGetErrorString(cudaGetLastError()));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float ms;
    for (int which = 0; which < 2; which++) {
        cudaEventRecord(e0);
        for (int r = 0; r < 200; r++) {
            if (which) k_v2_256<<<1, 256, smem3>>>(dt, n, dout, dinfo);
            else k_v2<<<1, SEQSUM2_THREADS, smem2>>>(dt, n, dout, dinfo);
        }
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        cudaEventElapsedTime(&ms, e0, e1);
        printf("%s: %.2f us per launch (back-to-back launches, includes ~2 us launch overhead)\n", which ? "v2 (256 threads)" : "v2", ms * 1000.f / 200);
    }
    return bad != 0;
}
