// mulcs_peak.cu -- does an IMAD.WIDE.U32 that only WRITES a carry predicate issue at the plain rate (2 cycles per
// warp instruction and scheduler) or at the carry-in (.X) rate (4 cycles)?  And what does a field multiplication
// built on carry-out-only MACs (mul_cs.cuh) reach against the shipped carry-chain one?  One JSON object on stdout.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include "../elliptic_b200/csrc/ecdsa_k256_body.cuh"
#include "../elliptic_b200/csrc/mul_cs.cuh"
using namespace eb;
#define ITERS 4096

__global__ void k_wide(u32* out, u32 seed) {
  u32 a = seed + threadIdx.x, b = seed * 3 + blockIdx.x + threadIdx.x * 7;
  u64 x[8];
  for (int i = 0; i < 8; i++) x[i] = a * (i + 1);
  for (int it = 0; it < ITERS; it++) {
#pragma unroll
    for (int r = 0; r < 4; r++) {
#pragma unroll
      for (int i = 0; i < 8; i++) asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(x[i]) : "r"(a), "r"(b));
    }
  }
  u64 s = 0;
  for (int i = 0; i < 8; i++) s ^= x[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = (u32)s ^ (u32)(s >> 32);
}
// carry-out only, each carry counted by one add-with-carry on the ALU pipe
__global__ void k_wide_co(u32* out, u32 seed) {
  u32 a = seed + threadIdx.x, b = seed * 3 + blockIdx.x + threadIdx.x * 7;
  u32 lo[8], hi[8], cn[8];
  for (int i = 0; i < 8; i++) { lo[i] = a * (i + 1); hi[i] = b + i; cn[i] = 0; }
  for (int it = 0; it < ITERS; it++) {
#pragma unroll
    for (int r = 0; r < 4; r++) {
#pragma unroll
      for (int i = 0; i < 8; i++)
        asm volatile("mad.lo.cc.u32 %0, %3, %4, %0; madc.hi.cc.u32 %1, %3, %4, %1; addc.u32 %2, %2, 0;"
                     : "+r"(lo[i]), "+r"(hi[i]), "+r"(cn[i]) : "r"(a), "r"(b));
    }
  }
  u32 s = 0;
  for (int i = 0; i < 8; i++) s ^= lo[i] ^ hi[i] ^ cn[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
// carry-in and carry-out (the shipped inner pattern)
__global__ void k_wide_cc(u32* out, u32 seed) {
  u32 a = seed + threadIdx.x, b = seed * 3 + blockIdx.x + threadIdx.x * 7;
  u32 x[16];
  for (int i = 0; i < 16; i++) x[i] = a * (i + 1);
  for (int it = 0; it < ITERS; it++) {
#pragma unroll
    for (int r = 0; r < 4; r++) {
      asm volatile("mad.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(x[0]), "+r"(x[1]) : "r"(a), "r"(b));
      asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(x[2]), "+r"(x[3]) : "r"(a), "r"(b));
      asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(x[4]), "+r"(x[5]) : "r"(a), "r"(b));
      asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.u32 %1, %2, %3, %1;" : "+r"(x[6]), "+r"(x[7]) : "r"(a), "r"(b));
      asm volatile("mad.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(x[8]), "+r"(x[9]) : "r"(b), "r"(a));
      asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(x[10]), "+r"(x[11]) : "r"(b), "r"(a));
      asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(x[12]), "+r"(x[13]) : "r"(b), "r"(a));
      asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.u32 %1, %2, %3, %1;" : "+r"(x[14]), "+r"(x[15]) : "r"(b), "r"(a));
    }
  }
  u32 s = 0;
  for (int i = 0; i < 16; i++) s ^= x[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__device__ __noinline__ fe fe_mul_cs(fe a, fe b) { u32 t[16]; mul_wide_cs<8>(t, a.v, b.v); fe r; fe_reduce512(r.v, t); return r; }
__device__ __noinline__ fe fe_sqr_cs(fe a) { u32 t[16]; sqr_wide_cs<8>(t, a.v); fe r; fe_reduce512(r.v, t); return r; }
__device__ __forceinline__ fe fe_mul_cs_inl(const fe& a, const fe& b) { u32 t[16]; mul_wide_cs<8>(t, a.v, b.v); fe r; fe_reduce512(r.v, t); return r; }
__device__ __forceinline__ fe fe_sqr_cs_inl(const fe& a) { u32 t[16]; sqr_wide_cs<8>(t, a.v); fe r; fe_reduce512(r.v, t); return r; }

// two independent products per call: half the call marshalling per product and two carry chains to interleave
struct fe_pair { fe a, b; };
__device__ __noinline__ fe_pair fe_mul2_call(fe a, fe b, fe c, fe d) { fe_pair r; r.a = fe_mul_inl(a, b); r.b = fe_mul_inl(c, d); return r; }
__device__ __noinline__ fe_pair fe_sqr2_call(fe a, fe c) { fe_pair r; r.a = fe_sqr_inl(a); r.b = fe_sqr_inl(c); return r; }

template <int OP>
__global__ void k_fe2(u32* out, u32 seed) {
  fe a, b, c, d;
  for (int i = 0; i < 8; i++) { a.v[i] = seed * (i + 1) + threadIdx.x; b.v[i] = seed * (i + 7) + blockIdx.x + 3 * threadIdx.x; c.v[i] = a.v[i] ^ 0x5555; d.v[i] = b.v[i] + 77; }
  for (int it = 0; it < ITERS / 4; it++) {
    if (OP == 0) { fe_pair r = fe_mul2_call(a, b, c, d); a = r.a; c = r.b; r = fe_mul2_call(b, a, d, c); b = r.a; d = r.b; }
    if (OP == 1) { fe_pair r = fe_sqr2_call(a, c); a = r.a; c = r.b; r = fe_sqr2_call(b, d); b = r.a; d = r.b; }
    if (OP == 2) { a = fe_mul(a, b); c = fe_mul(c, d); b = fe_mul(b, a); d = fe_mul(d, c); }          // same work, four calls
    if (OP == 3) { a = fe_mul_inl(a, b); c = fe_mul_inl(c, d); b = fe_mul_inl(b, a); d = fe_mul_inl(d, c); }
  }
  u32 s = 0;
  for (int i = 0; i < 8; i++) s ^= a.v[i] ^ b.v[i] ^ c.v[i] ^ d.v[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <int OP>
__global__ void k_fe(u32* out, u32 seed) {
  fe a, b;
  for (int i = 0; i < 8; i++) { a.v[i] = seed * (i + 1) + threadIdx.x; b.v[i] = seed * (i + 7) + blockIdx.x + 3 * threadIdx.x; }
  for (int it = 0; it < ITERS / 4; it++) {
    if (OP == 0) { a = fe_mul(a, b); b = fe_mul(b, a); }
    if (OP == 1) { a = fe_sqr(a); b = fe_sqr(b); }
    if (OP == 2) { a = fe_mul_cs(a, b); b = fe_mul_cs(b, a); }
    if (OP == 3) { a = fe_sqr_cs(a); b = fe_sqr_cs(b); }
    if (OP == 4) { a = fe_mul_cs_inl(a, b); b = fe_mul_cs_inl(b, a); }
    if (OP == 5) { a = fe_sqr_cs_inl(a); b = fe_sqr_cs_inl(b); }
    if (OP == 6) { a = fe_mul_inl(a, b); b = fe_mul_inl(b, a); }
    if (OP == 7) { a = fe_sqr_inl(a); b = fe_sqr_inl(b); }
  }
  u32 s = 0;
  for (int i = 0; i < 8; i++) s ^= a.v[i] ^ b.v[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// correctness on the device: carry-save products against the shipped ones on pseudo-random and edge operands
__global__ void k_check(unsigned long long* bad, u32 seed) {
  u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  fe a, b;
  u32 s = seed + i * 2654435761u;
  for (int k = 0; k < 8; k++) {
    s = s * 1664525u + 1013904223u; a.v[k] = s;
    s = s * 1664525u + 1013904223u; b.v[k] = s;
    if ((i & 7) == 1) a.v[k] = 0xffffffffu;
    if ((i & 7) == 2) { a.v[k] = 0xffffffffu; b.v[k] = 0xffffffffu; }
    if ((i & 7) == 3 && (k & 1)) b.v[k] = 0;
  }
  u32 t0[16], t1[16];
  mul_wide<8>(t0, a.v, b.v); mul_wide_cs<8>(t1, a.v, b.v);
  bool ok = true;
  for (int k = 0; k < 16; k++) ok = ok && t0[k] == t1[k];
  mul_wide<8>(t0, a.v, a.v); sqr_wide_cs<8>(t1, a.v);
  for (int k = 0; k < 16; k++) ok = ok && t0[k] == t1[k];
  if (!ok) atomicAdd(bad, 1ull);
}

template <typename K>
double run(K kern, int blocks, int threads, u32* d_out) {
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  kern<<<blocks, threads>>>(d_out, 12345u);
  cudaDeviceSynchronize();
  double best = 1e30;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0);
    kern<<<blocks, threads>>>(d_out, 12345u + rep);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  return best * 1e-3;
}

int main() {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, 0) != cudaSuccess) { printf("{\"error\": \"no device\"}\n"); return 1; }
  int sms = prop.multiProcessorCount;
  u32* d_out;
  cudaMalloc(&d_out, (size_t)sms * 64 * 1024 * 4);
  unsigned long long* d_bad; unsigned long long bad = 0;
  cudaMalloc(&d_bad, 8); cudaMemset(d_bad, 0, 8);
  k_check<<<4096, 256>>>(d_bad, 99u);
  cudaMemcpy(&bad, d_bad, 8, cudaMemcpyDeviceToHost);
  printf("{\"gpu\": \"%s\", \"sms\": %d, \"clock_khz\": %d, \"cs_mismatches_of_1048576\": %llu", prop.name, sms, prop.clockRate, bad);
  int cfgs[][2] = {{3, 128}, {4, 128}, {4, 256}, {2, 512}};
  for (auto& c : cfgs) {
    int blocks = sms * c[0], threads = c[1];
    double n = (double)blocks * threads, t;
    t = run(k_wide, blocks, threads, d_out);
    printf(",\n \"wide_%dx%d_Tmac\": %.3f", c[0], c[1], n * ITERS * 32 / t / 1e12);
    t = run(k_wide_co, blocks, threads, d_out);
    printf(", \"wide_carryout_counted_%dx%d_Tmac\": %.3f", c[0], c[1], n * ITERS * 32 / t / 1e12);
    t = run(k_wide_cc, blocks, threads, d_out);
    printf(", \"wide_cc_%dx%d_Tmac\": %.3f", c[0], c[1], n * ITERS * 32 / t / 1e12);
    const char* nm[8] = {"fe_mul", "fe_sqr", "fe_mul_cs", "fe_sqr_cs", "fe_mul_cs_inl", "fe_sqr_cs_inl", "fe_mul_inl", "fe_sqr_inl"};
    double ts[8];
    ts[0] = run(k_fe<0>, blocks, threads, d_out); ts[1] = run(k_fe<1>, blocks, threads, d_out);
    ts[2] = run(k_fe<2>, blocks, threads, d_out); ts[3] = run(k_fe<3>, blocks, threads, d_out);
    ts[4] = run(k_fe<4>, blocks, threads, d_out); ts[5] = run(k_fe<5>, blocks, threads, d_out);
    ts[6] = run(k_fe<6>, blocks, threads, d_out); ts[7] = run(k_fe<7>, blocks, threads, d_out);
    for (int k = 0; k < 8; k++) printf(", \"%s_%dx%d_G\": %.2f", nm[k], c[0], c[1], n * (ITERS / 4) * 2 / ts[k] / 1e9);
    const char* nm2[4] = {"fe_mul2_call", "fe_sqr2_call", "fe_mul_x4_calls", "fe_mul_x4_inl"};
    double t2[4] = {run(k_fe2<0>, blocks, threads, d_out), run(k_fe2<1>, blocks, threads, d_out), run(k_fe2<2>, blocks, threads, d_out), run(k_fe2<3>, blocks, threads, d_out)};
    for (int k = 0; k < 4; k++) printf(", \"%s_%dx%d_G\": %.2f", nm2[k], c[0], c[1], n * (ITERS / 4) * 4 / t2[k] / 1e9);
  }
  printf("}\n");
  return 0;
}
