// fp64.cu -- what the B200 FP64 pipe sustains, in the style of pipes.cu: issue cost (SMSP cycles per
// warp-instruction) of DFMA / DMUL / DADD at 1 - 4 warps per sub-partition, co-issue of DFMA with the integer
// pipes (IMAD on the FMA pipe's integer half, LOP3 on the ALU pipe), and the L2 read bandwidth an SM gets from a
// 64 MB buffer that is already resident in the 126 MB L2.  One CTA per SM, 32 x w threads per sub-partition.
// Question it answers: can a float64 FFT external product run at >= 1 FP64 warp-instruction per clock per SM?
#include <cstdio>
#include <cuda_runtime.h>
#define REP8(X) X X X X X X X X
#define REP64(X) REP8(REP8(X))
typedef unsigned u32;

// 8 independent accumulator chains per copy, two copies: 16 in flight, enough to cover the DFMA latency at 1 warp
#define F8(OP) asm volatile(OP " %0, %0, %8, %9;\n\t" OP " %1, %1, %8, %9;\n\t" OP " %2, %2, %8, %9;\n\t" OP " %3, %3, %8, %9;\n\t" \
                            OP " %4, %4, %8, %9;\n\t" OP " %5, %5, %8, %9;\n\t" OP " %6, %6, %8, %9;\n\t" OP " %7, %7, %8, %9;" \
                            : "+d"(x0), "+d"(x1), "+d"(x2), "+d"(x3), "+d"(x4), "+d"(x5), "+d"(x6), "+d"(x7) : "d"(m), "d"(c));
#define F8B(OP) asm volatile(OP " %0, %0, %8, %9;\n\t" OP " %1, %1, %8, %9;\n\t" OP " %2, %2, %8, %9;\n\t" OP " %3, %3, %8, %9;\n\t" \
                             OP " %4, %4, %8, %9;\n\t" OP " %5, %5, %8, %9;\n\t" OP " %6, %6, %8, %9;\n\t" OP " %7, %7, %8, %9;" \
                             : "+d"(y0), "+d"(y1), "+d"(y2), "+d"(y3), "+d"(y4), "+d"(y5), "+d"(y6), "+d"(y7) : "d"(m), "d"(c));
#define M8(OP) asm volatile(OP " %0, %0, %8;\n\t" OP " %1, %1, %8;\n\t" OP " %2, %2, %8;\n\t" OP " %3, %3, %8;\n\t" \
                            OP " %4, %4, %8;\n\t" OP " %5, %5, %8;\n\t" OP " %6, %6, %8;\n\t" OP " %7, %7, %8;" \
                            : "+d"(x0), "+d"(x1), "+d"(x2), "+d"(x3), "+d"(x4), "+d"(x5), "+d"(x6), "+d"(x7) : "d"(m));
#define M8B(OP) asm volatile(OP " %0, %0, %8;\n\t" OP " %1, %1, %8;\n\t" OP " %2, %2, %8;\n\t" OP " %3, %3, %8;\n\t" \
                             OP " %4, %4, %8;\n\t" OP " %5, %5, %8;\n\t" OP " %6, %6, %8;\n\t" OP " %7, %7, %8;" \
                             : "+d"(y0), "+d"(y1), "+d"(y2), "+d"(y3), "+d"(y4), "+d"(y5), "+d"(y6), "+d"(y7) : "d"(m));
#define I4 asm volatile("mad.lo.u32 %0, %0, %1, %2; mad.lo.u32 %1, %1, %2, %3; mad.lo.u32 %2, %2, %3, %0; mad.lo.u32 %3, %3, %0, %1;" : "+r"(a), "+r"(b), "+r"(cc), "+r"(d));
#define L4 asm volatile("xor.b32 %0, %0, %1; xor.b32 %1, %1, %2; xor.b32 %2, %2, %3; xor.b32 %3, %3, %0;" : "+r"(a), "+r"(b), "+r"(cc), "+r"(d));

// 1: 16 DFMA   2: 16 DMUL   3: 16 DADD
// 4: 16 DFMA + 4 IMAD   5: 16 DFMA + 4 LOP3   6: 16 DFMA + 4 IMAD + 4 LOP3   7: 8 DFMA + 4 IMAD + 4 LOP3
// 8: 4 IMAD + 4 LOP3 alone (the integer part of 6 and 7)
template <int MODE> __global__ void __launch_bounds__(1024) kern(u32 *out, double *dout, int iters, long long *cycles)
{
    const double m = 0.9999999 + 1e-12 * threadIdx.x, c = 1e-9;
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    double y0 = x0 + 8, y1 = x0 + 9, y2 = x0 + 10, y3 = x0 + 11, y4 = x0 + 12, y5 = x0 + 13, y6 = x0 + 14, y7 = x0 + 15;
    u32 a = threadIdx.x + out[0], b = a + 1, cc = a + 2, d = a + 3;
    __syncthreads();
    long long t0 = clock64();
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
        if (MODE == 1) { REP64(F8("fma.rn.f64") F8B("fma.rn.f64")) }
        if (MODE == 2) { REP64(M8("mul.rn.f64") M8B("mul.rn.f64")) }
        if (MODE == 3) { REP64(M8("add.rn.f64") M8B("add.rn.f64")) }
        if (MODE == 4) { REP64(F8("fma.rn.f64") I4 F8B("fma.rn.f64")) }
        if (MODE == 5) { REP64(F8("fma.rn.f64") L4 F8B("fma.rn.f64")) }
        if (MODE == 6) { REP64(F8("fma.rn.f64") I4 F8B("fma.rn.f64") L4) }
        if (MODE == 7) { REP64(F8("fma.rn.f64") I4 L4) }
        if (MODE == 8) { REP64(I4 L4) }
    }
    long long t1 = clock64();
    dout[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7 + y0 + y1 + y2 + y3 + y4 + y5 + y6 + y7;
    out[1 + blockIdx.x * blockDim.x + threadIdx.x] = a ^ b ^ cc ^ d;
    if (threadIdx.x == 0 && blockIdx.x == 0) *cycles = t1 - t0;
}

template <int MODE> void run(const char *name, int fp64_per_block, int sms, u32 *out, double *dout, long long *dcyc)
{
    for (int w : {1, 2, 3, 4}) {
        const int iters = 256;
        kern<MODE><<<sms, w * 128>>>(out, dout, iters, dcyc);
        cudaDeviceSynchronize();
        kern<MODE><<<sms, w * 128>>>(out, dout, iters, dcyc);
        cudaDeviceSynchronize();
        long long cyc;
        cudaMemcpy(&cyc, dcyc, 8, cudaMemcpyDeviceToHost);
        // SMSP cycles per repetition of the block per warp; FP64 warp-instructions per clock per SM = 4 SMSPs x
        // w warps x fp64_per_block / cycles of one repetition
        const double per_block = (double)cyc / (iters * 64.0 * w);
        printf("mode %d %-36s warps/SMSP=%d  cycles per block per warp = %6.2f   FP64 warp-instr / clk / SM = %.3f\n", MODE,
               name, w, per_block, fp64_per_block ? 4.0 * fp64_per_block / per_block : 0.0);
    }
}

// L2 read bandwidth: a 64 MB buffer is read once (now L2-resident), then every CTA streams its own slice of it
// `passes` times with 16-byte ld.global.cg (L2, not L1); bytes / kernel time (CUDA events)
__global__ void __launch_bounds__(1024) l2_read(const int4 *__restrict__ buf, size_t n16, int passes, int4 *sink)
{
    int4 acc = make_int4(0, 0, 0, 0);
    const size_t per = n16 / gridDim.x, base = blockIdx.x * per;
    for (int p = 0; p < passes; p++)
        for (size_t i = threadIdx.x; i < per; i += blockDim.x) {
            const int4 v = __ldcg(buf + base + ((i + (size_t)p * 4096) % per));
            acc.x ^= v.x; acc.y ^= v.y; acc.z ^= v.z; acc.w ^= v.w;
        }
    if (acc.x == 0x12345678 && acc.y == 0x9abcdef) sink[threadIdx.x] = acc;
}

int main()
{
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, 0);
    int clk_khz = 0;
    cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0);
    const int sms = prop.multiProcessorCount;
    printf("device %s, %d SMs, L2 %d MB, max SM clock %d MHz\n", prop.name, sms, prop.l2CacheSize >> 20, clk_khz / 1000);
    u32 *out; double *dout; long long *dcyc;
    cudaMalloc(&out, (sms * 1024 + 1) * 4); cudaMemset(out, 0, (sms * 1024 + 1) * 4);
    cudaMalloc(&dout, sms * 1024 * 8); cudaMalloc(&dcyc, 8);
    run<1>("16 DFMA", 16, sms, out, dout, dcyc);
    run<2>("16 DMUL", 16, sms, out, dout, dcyc);
    run<3>("16 DADD", 16, sms, out, dout, dcyc);
    run<4>("16 DFMA + 4 IMAD", 16, sms, out, dout, dcyc);
    run<5>("16 DFMA + 4 LOP3", 16, sms, out, dout, dcyc);
    run<6>("16 DFMA + 4 IMAD + 4 LOP3", 16, sms, out, dout, dcyc);
    run<7>("8 DFMA + 4 IMAD + 4 LOP3", 8, sms, out, dout, dcyc);
    run<8>("4 IMAD + 4 LOP3", 0, sms, out, dout, dcyc);

    const size_t bytes = 64ull << 20, n16 = bytes / 16;
    int4 *buf, *sink;
    cudaMalloc(&buf, bytes); cudaMalloc(&sink, 1024 * 16);
    cudaMemset(buf, 1, bytes);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int threads : {256, 512, 1024}) {
        const int passes = 20;
        l2_read<<<sms, threads>>>(buf, n16, 1, sink);      // warm: the buffer is resident in L2 afterwards
        cudaEventRecord(e0);
        l2_read<<<sms, threads>>>(buf, n16, passes, sink);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        const double gbs = (double)bytes * passes / (ms * 1e-3) / 1e9;
        printf("L2 read, 64 MB resident, %4d threads/SM: %.0f GB/s total, %.1f GB/s per SM, %.1f B/clk/SM at %d MHz\n",
               threads, gbs, gbs / sms, gbs * 1e9 / sms / (clk_khz * 1e3), clk_khz / 1000);
    }
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(err)); return 1; }
    return 0;
}
