// in_range_math_check.cu - compares sqrt_in_range / div_in_range / atan2_deg<true> (csrc/s2d_math.cuh) with the IEEE
// operators they stand in for, bit for bit, over the operand domains in_range_vector proves (tests/test_gpu_in_range_math.py
// builds and runs it).  Prints "<name> <cases> <mismatches>" per check and the first mismatch, then the division's
// mismatches just outside its domain and how many vectors in_range_vector sent to the guard-free forms.
#include <cstdio>
#include <cstdint>
#include <cstring>

#include "s2d_math.cuh"

using namespace s2d;

__device__ unsigned long long g_bad[3];
__device__ unsigned long long g_cases[3];
__device__ float g_first[3][3];
__device__ unsigned long long g_outside, g_outside_cases, g_fast;

__device__ void report(int which, float a, float b, bool bad) {
  if (bad) {
    const unsigned long long k = atomicAdd(&g_bad[which], 1ull);
    if (k == 0) {
      g_first[which][0] = a;
      g_first[which][1] = b;
    }
  }
}

__device__ uint32_t mix(uint32_t x) {  // lowbias32
  x ^= x >> 16;
  x *= 0x7feb352du;
  x ^= x >> 15;
  x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}

// every float in [2^-40, 2^40]
__global__ void check_sqrt(uint32_t lo_bits, uint32_t count) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < count; j += gridDim.x * blockDim.x) {
    const float x = __uint_as_float(lo_bits + j);
    const float got = sqrt_in_range(x), want = sqrtf(x);
    report(0, x, 0.0f, __float_as_uint(got) != __float_as_uint(want));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&g_cases[0], count);
}

// divisors: every 64th float of [2^-21, 2^22] and both ends.  Per divisor b, inside div_in_range's domain (a = +0 or
// 2^-100 <= |a| <= b): +0, +-b, the floats next to +-b, +-2^-100 and the float above it, b / 2, and 22 numerators with
// random bits (uniform in exponent).  Outside it (counted apart, not required to match): -0, the smallest normal and
// subnormal numerators, and numerators with random bits below 2^-100.
__device__ float random_below(uint32_t r, uint32_t top_exp) {  // random bits, biased exponent in [0, top_exp)
  const uint32_t m = ((r % top_exp) << 23) | (mix(r) & 0x7fffffu);
  return (r & 0x80000000u) ? -__uint_as_float(m) : __uint_as_float(m);
}
__global__ void check_div(uint32_t lo_bits, uint32_t hi_bits) {
  const uint32_t ndiv = (hi_bits - lo_bits) / 64 + 2;
  const uint32_t e_min = __float_as_uint(kInRangeMinComponent) >> 23;
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < ndiv; j += gridDim.x * blockDim.x) {
    const float b = __uint_as_float(j == ndiv - 1 ? hi_bits : lo_bits + 64 * j);
    const uint32_t bb = __float_as_uint(b), eb = bb >> 23;
    const float m = kInRangeMinComponent, m1 = __uint_as_float(__float_as_uint(kInRangeMinComponent) + 1);
    float in[32] = {0.0f, b, -b, __uint_as_float(bb - 1), -__uint_as_float(bb - 1), m, -m, m1, -m1, 0.5f * b};
    for (int t = 10; t < 32; ++t) {
      const uint32_t r = mix(j * 64u + t);
      float a = random_below(r, eb - e_min + 1);
      a = __uint_as_float(__float_as_uint(a) + (e_min << 23));  // exponent in [e_min, eb]
      in[t] = fabsf(a) > b ? copysignf(b, a) : a;
    }
    for (int t = 0; t < 32; ++t) report(1, in[t], b, __float_as_uint(div_in_range(in[t], b)) != __float_as_uint(in[t] / b));
    atomicAdd(&g_cases[1], 32ull);
    float out[8] = {-0.0f, 1.17549435e-38f, -1.17549435e-38f, 1.4e-45f, -1.4e-45f};
    for (int t = 5; t < 8; ++t) out[t] = random_below(mix(j * 64u + 40u + t), e_min);
    for (int t = 0; t < 8; ++t)
      if (__float_as_uint(div_in_range(out[t], b)) != __float_as_uint(out[t] / b)) atomicAdd(&g_outside, 1ull);
    atomicAdd(&g_outside_cases, 8ull);
  }
}

// 2^28 vectors with random bits, components from 2^-150 (subnormal) to 2^24 and axis-aligned ones, through
// check_episode's selection: in_range_vector -> atan2_deg<true> and sqrt_in_range, else the IEEE forms.  Compared with
// atan2_deg and sqrtf; g_fast counts the vectors that took the guard-free forms.
__global__ void check_atan2(uint32_t n) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const uint32_t r = mix(j), r2 = mix(r ^ 0x9e3779b9u);
    float x = __uint_as_float(((107u + r % 43u) << 23) | (r2 & 0x7fffffu));
    float y = __uint_as_float(((r2 >> 24) % 4u == 0) ? 0u : (((mix(r2) % 152u) << 23) | (mix(r2 + 1) & 0x7fffffu)));
    if (r & 1u) x = -x;
    if (r & 2u) y = -y;
    if (r & 4u) {
      const float t = x;
      x = y;
      y = t;
    }
    const float d2 = x * x + y * y;
    const bool fast = in_range_vector(x, y, d2);
    const float got = fast ? atan2_deg<true>(y, x) : atan2_deg(y, x), want = atan2_deg(y, x);
    const float dist = fast ? sqrt_in_range(d2) : sqrtf(d2);
    report(2, y, x, __float_as_uint(got) != __float_as_uint(want) || __float_as_uint(dist) != __float_as_uint(sqrtf(d2)));
    if (fast) atomicAdd(&g_fast, 1ull);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&g_cases[2], n);
}

int main() {
  uint32_t lo, hi;
  const float d2lo = kInRangeD2Min, d2hi = kInRangeD2Max, blo = 0x1p-21f, bhi = 0x1p22f;
  memcpy(&lo, &d2lo, 4);
  memcpy(&hi, &d2hi, 4);
  check_sqrt<<<4096, 256>>>(lo, hi - lo + 1);
  memcpy(&lo, &blo, 4);
  memcpy(&hi, &bhi, 4);
  check_div<<<4096, 256>>>(lo, hi);
  check_atan2<<<4096, 256>>>(1u << 28);
  const cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    printf("cuda error %s\n", cudaGetErrorString(e));
    return 1;
  }
  unsigned long long bad[3], cases[3];
  float first[3][3];
  cudaMemcpyFromSymbol(bad, g_bad, sizeof(bad));
  cudaMemcpyFromSymbol(cases, g_cases, sizeof(cases));
  cudaMemcpyFromSymbol(first, g_first, sizeof(first));
  unsigned long long outside, outside_cases, fast;
  cudaMemcpyFromSymbol(&outside, g_outside, sizeof(outside));
  cudaMemcpyFromSymbol(&outside_cases, g_outside_cases, sizeof(outside_cases));
  cudaMemcpyFromSymbol(&fast, g_fast, sizeof(fast));
  const char* names[3] = {"sqrt", "div", "atan2"};
  for (int i = 0; i < 3; ++i) {
    printf("%s %llu %llu\n", names[i], cases[i], bad[i]);
    if (bad[i]) printf("  first mismatch: %a %a\n", first[i][0], first[i][1]);
  }
  printf("div_outside_domain %llu %llu\n", outside_cases, outside);
  printf("atan2_fast %llu\n", fast);
  return 0;
}
