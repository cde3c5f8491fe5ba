// bench_pipes.cu -- issue rate of the SASS operations the interpreter is made of, on the GPU it runs on.
//
// Which execution pipe an integer operation goes to, and at what rate, decides how many cycles an emulated instruction
// costs (DESIGN.md 4.1): the single-lane interpreter is bound by its integer-ALU-pipe instructions.  For each operation a
// kernel runs a long unrolled stream of it: 8 independent chains per thread (each step reads the previous value of its own
// and of the next chain, so nothing folds away), 1,024 threads per block, one block per SM.  Thread 0 of every block reads
// the SM clock around the stream; the result is warp instructions per cycle per SM (4 = one per cycle on each of the four
// schedulers).  A second set of streams mixes each operation 1:1 with LOP3: if the two share a pipe the mix runs at that
// pipe's rate, if not it runs faster.  tools/bench_pipes.py compiles this file, checks in the SASS that each stream contains
// the intended operation, runs it and writes the JSON record.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#define CHAINS 8
#define UNROLL 16
#define ITERS 2048
#define THREADS 1024

__constant__ uint32_t c_tab[256];  // LDC stream: entry i = byte offset of entry (i * 7 + 1) & 255

// A chain of immediate adds or of multiplications by a power of two folds into one operation, so VIADD and IMAD.SHL are
// only measured in the mixes (whose LOP3 sits between two of them).
// one step of every chain: x[i] = OP(x[i], x[(i + 1) % CHAINS]); y is a per-thread value the compiler does not know
#define STEP(OP)                                                   \
    _Pragma("unroll") for (int i = 0; i < CHAINS; i++) {          \
        const uint32_t a = x[i], b = x[(i + 1) % CHAINS];          \
        (void)a; (void)b; (void)y;                                 \
        OP;                                                        \
    }

#define OP_LOP3 asm volatile("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(x[i]) : "r"(a), "r"(b), "r"(y))
#define OP_SHF asm volatile("shf.l.wrap.b32 %0, %1, %2, %3;" : "=r"(x[i]) : "r"(a), "r"(b), "r"(y))
#define OP_PRMT asm volatile("prmt.b32 %0, %1, %2, %3;" : "=r"(x[i]) : "r"(a), "r"(b), "r"(y))
#define OP_IADD3 asm volatile("{\n\t.reg .u32 t;\n\tadd.u32 t, %1, %2;\n\tadd.u32 %0, t, %3;\n\t}" : "=r"(x[i]) : "r"(a), "r"(b), "r"(y))
#define OP_SEL asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\tselp.b32 %0, %1, %2, p;\n\t}" : "=r"(x[i]) : "r"(a), "r"(b), "r"(y))
// ISETP: a compare whose result feeds the next compare of the chain through its predicate input (setp.xor), 8 in one block
#define OP_ISETP                                                                                                   \
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %0, 0;\n\tsetp.lt.u32.xor q, %1, %2, p;\n\t"            \
                 "setp.lt.u32.xor p, %2, %1, q;\n\tsetp.gt.u32.xor q, %1, %3, p;\n\tsetp.gt.u32.xor p, %3, %2, q;\n\t" \
                 "setp.le.u32.xor q, %1, %2, p;\n\tsetp.le.u32.xor p, %2, %3, q;\n\tsetp.ge.u32.xor q, %3, %1, p;\n\t"  \
                 "setp.ge.u32.xor p, %1, %3, q;\n\tselp.b32 %0, %1, %2, p;\n\t}"                                      \
                 : "+r"(x[i]) : "r"(a), "r"(b), "r"(y))
#define OP_LEA asm volatile("{\n\t.reg .u32 t;\n\tshl.b32 t, %1, 3;\n\tadd.u32 %0, t, %2;\n\t}" : "=r"(x[i]) : "r"(a), "r"(b))
#define OP_VIADD asm volatile("add.u32 %0, %1, 0x1234567;" : "=r"(x[i]) : "r"(b))
#define OP_IMAD asm volatile("mad.lo.u32 %0, %1, %2, %3;" : "=r"(x[i]) : "r"(a), "r"(b), "r"(y))
#define OP_IMAD_SHL asm volatile("mul.lo.u32 %0, %1, 8;" : "=r"(x[i]) : "r"(b))
#define OP_IMAD_IADD asm volatile("add.u32 %0, %1, %2;" : "=r"(x[i]) : "r"(a), "r"(b))
// table streams chase byte offsets: every chain value is a multiple of 4 below 1,024 (the mixes' LOP3 keeps it so) and the
// same in all lanes of a warp (chains and y start from the warp index), as in the single-lane interpreter, which reads its
// tables with one address per warp: a constant-cache read with 32 different addresses is serialised
#define OP_LDC x[i] = *(const uint32_t *)((const char *)c_tab + a)
#define OP_LDS x[i] = *(volatile uint32_t *)((char *)s_tab + a)
#define OP_MIX(OP) \
    OP;            \
    asm volatile("lop3.b32 %0, %1, 0x3FC, %2, 0x48;" : "=r"(x[(i + 4) % CHAINS]) : "r"(x[(i + 4) % CHAINS]), "r"(y))

#define KERNEL(NAME, OP)                                                                                   \
    __global__ void __launch_bounds__(THREADS) k_##NAME(uint32_t seed, uint32_t *sink, long long *cycles) { \
        __shared__ uint32_t s_tab[256];                                                                    \
        s_tab[threadIdx.x & 255] = (((threadIdx.x & 255) * 7 + 1) & 255) * 4;                               \
        __syncthreads();                                                                                   \
        const uint32_t y = seed ^ (threadIdx.x / 32);                                                      \
        uint32_t x[CHAINS];                                                                                \
        _Pragma("unroll") for (int i = 0; i < CHAINS; i++) x[i] = (seed * (i + 3) + (threadIdx.x / 32) * 4) & 0x3FC; \
        __syncthreads();                                                                                   \
        const long long t0 = clock64();                                                                    \
        for (int it = 0; it < ITERS; it++) {                                                               \
            _Pragma("unroll") for (int u = 0; u < UNROLL; u++) { STEP(OP) }                                \
        }                                                                                                  \
        __syncthreads();                                                                                   \
        const long long t1 = clock64();                                                                    \
        uint32_t r = 0;                                                                                    \
        _Pragma("unroll") for (int i = 0; i < CHAINS; i++) r ^= x[i];                                      \
        if (r == 0x9E3779B9u) sink[0] = r;                                                                 \
        if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;                                                \
    }

KERNEL(LOP3, OP_LOP3)
KERNEL(SHF, OP_SHF)
KERNEL(PRMT, OP_PRMT)
KERNEL(IADD3, OP_IADD3)
KERNEL(SEL, OP_SEL)
KERNEL(ISETP, OP_ISETP)
KERNEL(LEA, OP_LEA)
KERNEL(IMAD, OP_IMAD)
KERNEL(IMAD_IADD, OP_IMAD_IADD)
KERNEL(LDC, OP_LDC)
KERNEL(LDS, OP_LDS)
KERNEL(MIX_SHF, OP_MIX(OP_SHF))
KERNEL(MIX_PRMT, OP_MIX(OP_PRMT))
KERNEL(MIX_IADD3, OP_MIX(OP_IADD3))
KERNEL(MIX_SEL, OP_MIX(OP_SEL))
KERNEL(MIX_ISETP, OP_MIX(OP_ISETP))
KERNEL(MIX_LEA, OP_MIX(OP_LEA))
KERNEL(MIX_VIADD, OP_MIX(OP_VIADD))
KERNEL(MIX_IMAD, OP_MIX(OP_IMAD))
KERNEL(MIX_IMAD_SHL, OP_MIX(OP_IMAD_SHL))
KERNEL(MIX_IMAD_IADD, OP_MIX(OP_IMAD_IADD))
KERNEL(MIX_LDC, OP_MIX(OP_LDC))
KERNEL(MIX_LDS, OP_MIX(OP_LDS))

typedef void (*kfn)(uint32_t, uint32_t *, long long *);
struct Entry { const char *name; kfn k; int ops_per_step; };  // ops_per_step: stream instructions per chain step (the mix: + 1 LOP3; ISETP: 8 compares, the SEL and the ISETP that
// turns the chain's register into a predicate)
static const Entry kEntries[] = {
    {"LOP3", k_LOP3, 1}, {"SHF", k_SHF, 1}, {"PRMT", k_PRMT, 1}, {"IADD3", k_IADD3, 1}, {"SEL", k_SEL, 1},
    {"ISETP", k_ISETP, 10}, {"LEA", k_LEA, 1}, {"IMAD", k_IMAD, 1}, 
    {"IMAD_IADD", k_IMAD_IADD, 1}, {"LDC", k_LDC, 1}, {"LDS", k_LDS, 1},
    {"MIX_SHF", k_MIX_SHF, 2}, {"MIX_PRMT", k_MIX_PRMT, 2}, {"MIX_IADD3", k_MIX_IADD3, 2}, {"MIX_SEL", k_MIX_SEL, 2},
    {"MIX_ISETP", k_MIX_ISETP, 11}, {"MIX_LEA", k_MIX_LEA, 2}, {"MIX_VIADD", k_MIX_VIADD, 2}, {"MIX_IMAD", k_MIX_IMAD, 2},
    {"MIX_IMAD_SHL", k_MIX_IMAD_SHL, 2}, {"MIX_IMAD_IADD", k_MIX_IMAD_IADD, 2}, {"MIX_LDC", k_MIX_LDC, 2}, {"MIX_LDS", k_MIX_LDS, 2},
};

#define CK(x)                                                                      \
    do {                                                                           \
        cudaError_t e_ = (x);                                                      \
        if (e_ != cudaSuccess) {                                                   \
            fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); \
            return 1;                                                              \
        }                                                                          \
    } while (0)

// prints one line per stream: name, warp instructions per cycle per SM (median over the SMs of the best of 3 launches)
int main() {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    const int sms = prop.multiProcessorCount;
    uint32_t tab[256];
    for (int i = 0; i < 256; i++) tab[i] = ((i * 7 + 1) & 255) * 4;
    CK(cudaMemcpyToSymbol(c_tab, tab, sizeof(tab)));
    uint32_t *sink;
    long long *cyc;
    CK(cudaMalloc(&sink, 4));
    CK(cudaMalloc(&cyc, sizeof(long long) * sms));
    long long *h = new long long[sms];
    printf("device %s sms %d\n", prop.name, sms);
    for (const Entry &en : kEntries) {
        double best = 0;
        for (int rep = 0; rep < 3; rep++) {
            en.k<<<sms, THREADS>>>(0x12345u + rep, sink, cyc);
            CK(cudaGetLastError());
            CK(cudaDeviceSynchronize());
            CK(cudaMemcpy(h, cyc, sizeof(long long) * sms, cudaMemcpyDeviceToHost));
            // median block
            for (int i = 1; i < sms; i++)
                for (int j = i; j > 0 && h[j - 1] > h[j]; j--) { long long t = h[j]; h[j] = h[j - 1]; h[j - 1] = t; }
            const double warp_instr = (double)(THREADS / 32) * ITERS * UNROLL * CHAINS * en.ops_per_step;
            const double rate = warp_instr / (double)h[sms / 2];
            if (rate > best) best = rate;
        }
        printf("%s %.4f\n", en.name, best);
    }
    delete[] h;
    return 0;
}
