"""Issue cost of packed single-precision FMA (FFMA2) against scalar FFMA on one SM.

Every thread of one block per SM runs a loop of fused multiply-adds on registers:
  * dependent:   one chain, each FMA waits for the previous one (latency);
  * independent: 8 chains interleaved (issue rate, with enough warps to hide latency).
The scalar form does one FFMA per element, the packed form one FFMA2 (__ffma2_rn) per PAIR of elements.  Reported
per SM: warp instructions per cycle and elements per cycle, from clock64() around the loop of every warp.  If FFMA2
issued at half the rate of FFMA (two issue slots each), packing would save no issue slots.

Compiles its kernel with nvcc into a temporary directory, checks the SASS for FFMA2, and prints one JSON line with the
GPU name, power limit and maximum SM clock read in the same run.

    python tools/ffma2_rate.py [--iters 4096] [--warps 1 2 4 8 16 32]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from goal_types_time import gpu_info  # noqa: E402

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SRC = r"""
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>

constexpr int CHAINS = 8;

// mode: 0 scalar dependent, 1 scalar independent, 2 packed dependent, 3 packed independent
template <int MODE>
__global__ void fma_loop(float* out, long long* cycles, int iters, float a, float b)
{
    float s[CHAINS], t[CHAINS];
    float2 p[CHAINS];
#pragma unroll
    for (int k = 0; k < CHAINS; ++k) {
        s[k] = threadIdx.x + k;
        t[k] = threadIdx.x - k;
        p[k] = make_float2(s[k], t[k]);
    }
    const float2 a2 = make_float2(a, a), b2 = make_float2(b, b);
    __syncthreads();
    const long long c0 = clock64();
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            if (MODE == 0) {
                // one chain of 2 * CHAINS FMAs (the same elements per loop trip as the independent form)
#pragma unroll
                for (int k = 0; k < 2 * CHAINS; ++k) s[0] = fmaf(s[0], a, b);
            } else if (MODE == 1) {
#pragma unroll
                for (int k = 0; k < CHAINS; ++k) { s[k] = fmaf(s[k], a, b); t[k] = fmaf(t[k], a, b); }
            } else if (MODE == 2) {
#pragma unroll
                for (int k = 0; k < CHAINS; ++k) p[0] = __ffma2_rn(p[0], a2, b2);
            } else {
#pragma unroll
                for (int k = 0; k < CHAINS; ++k) p[k] = __ffma2_rn(p[k], a2, b2);
            }
        }
    }
    const long long c1 = clock64();
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < CHAINS; ++k) acc += s[k] + t[k] + p[k].x + p[k].y;
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    if ((threadIdx.x & 31) == 0) cycles[blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32] = c1 - c0;
}

template <int MODE>
static void run(int sms, int warps, int iters, float* d_out, long long* d_cyc, long long* h_cyc)
{
    const int threads = 32 * warps;
    fma_loop<MODE><<<sms, threads>>>(d_out, d_cyc, iters, 0.999f, 1e-3f);   // warm-up
    fma_loop<MODE><<<sms, threads>>>(d_out, d_cyc, iters, 0.999f, 1e-3f);
    if (cudaDeviceSynchronize() != cudaSuccess) { fprintf(stderr, "kernel failed\n"); exit(1); }
    cudaMemcpy(h_cyc, d_cyc, sizeof(long long) * sms * warps, cudaMemcpyDeviceToHost);
    long long worst = 0;
    for (int i = 0; i < sms * warps; ++i) worst = h_cyc[i] > worst ? h_cyc[i] : worst;
    // warp instructions in the loop: MODE 0/1 issue 16 FFMA per trip, 2/3 issue 8 FFMA2 (16 elements either way)
    const double trips = (double)iters * 8.0;
    const double instr = trips * (MODE < 2 ? 16.0 : 8.0) * warps;   // per SM (one block per SM)
    const double elems = trips * 16.0 * 32.0 * warps;
    printf("{\"mode\": \"%s\", \"warps_per_sm\": %d, \"cycles\": %lld, \"warp_instr_per_cycle\": %.4f, "
           "\"elements_per_cycle\": %.2f}\n",
           MODE == 0 ? "ffma_dep" : MODE == 1 ? "ffma_indep" : MODE == 2 ? "ffma2_dep" : "ffma2_indep",
           warps, worst, instr / worst, elems / worst);
}

int main(int argc, char** argv)
{
    const int iters = atoi(argv[1]);
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    float* d_out;
    long long* d_cyc;
    cudaMalloc(&d_out, sizeof(float) * sms * 1024);
    cudaMalloc(&d_cyc, sizeof(long long) * sms * 32);
    long long* h_cyc = (long long*)malloc(sizeof(long long) * sms * 32);
    for (int a = 2; a < argc; ++a) {
        const int w = atoi(argv[a]);
        run<0>(sms, w, iters, d_out, d_cyc, h_cyc);
        run<1>(sms, w, iters, d_out, d_cyc, h_cyc);
        run<2>(sms, w, iters, d_out, d_cyc, h_cyc);
        run<3>(sms, w, iters, d_out, d_cyc, h_cyc);
    }
    cudaFree(d_out);
    cudaFree(d_cyc);
    free(h_cyc);
    return 0;
}
"""


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--iters", type=int, default=4096)
    ap.add_argument("--warps", type=int, nargs="+", default=[1, 2, 4, 8, 16, 32])
    ap.add_argument("--compile-only", action="store_true", help="build and check the SASS, do not run")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "ffma2_rate.cu")
        exe = os.path.join(tmp, "ffma2_rate")
        with open(src, "w") as f:
            f.write(SRC)
        subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe, src], check=True)
        sass = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", exe], check=True, capture_output=True,
                              text=True).stdout
        n_ffma2 = sum(1 for line in sass.splitlines() if "FFMA2" in line)
        if n_ffma2 == 0:
            raise SystemExit("no FFMA2 in the packed kernels' SASS")
        if args.compile_only:
            print(json.dumps({"ffma2_in_sass": n_ffma2}))
            return
        run = subprocess.run([exe, str(args.iters)] + [str(w) for w in args.warps], check=True, capture_output=True,
                             text=True)
    rows = [json.loads(line) for line in run.stdout.splitlines() if line.startswith("{")]
    print(json.dumps({"gpu": gpu_info(), "iters": args.iters, "ffma2_in_sass": n_ffma2, "rows": rows}))


if __name__ == "__main__":
    main()
