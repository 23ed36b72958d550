// elem_codec.cuh -- fp32 / bf16 / fp16 element loads and stores by dtype code (0 / 1 / 2, the codes of the C ABI), one
// element or 8 adjacent elements (one 16-byte vector for bf16 / fp16, two for fp32; the caller guarantees the alignment).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

template <int DT> struct ElemCodec;
template <> struct ElemCodec<0> {                    // fp32
  __device__ static float load(const void* p, size_t i) { return __ldg(reinterpret_cast<const float*>(p) + i); }
  __device__ static void load8(const void* p, size_t i, float (&f)[8]) {
    const float4* q = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + i);
    const float4 a = __ldg(q), b = __ldg(q + 1);
    f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
  }
  __device__ static void store(void* p, size_t i, float v) { reinterpret_cast<float*>(p)[i] = v; }
  __device__ static void store8(void* p, size_t i, const float (&o)[8]) {
    float4* q = reinterpret_cast<float4*>(reinterpret_cast<float*>(p) + i);
    q[0] = make_float4(o[0], o[1], o[2], o[3]); q[1] = make_float4(o[4], o[5], o[6], o[7]);
  }
};
template <> struct ElemCodec<1> {                    // bf16
  __device__ static float h2f(uint32_t u) { return __uint_as_float(u << 16); }
  __device__ static uint32_t f2h(float x) { __nv_bfloat16 h = __float2bfloat16_rn(x); return *reinterpret_cast<uint16_t*>(&h); }
  __device__ static float load(const void* p, size_t i) { return h2f(__ldg(reinterpret_cast<const uint16_t*>(p) + i)); }
  __device__ static void load8(const void* p, size_t i, float (&f)[8]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p) + i));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) { f[2 * e] = h2f(w[e] & 0xffffu); f[2 * e + 1] = h2f(w[e] >> 16); }
  }
  __device__ static void store(void* p, size_t i, float v) { reinterpret_cast<uint16_t*>(p)[i] = (uint16_t)f2h(v); }
  __device__ static void store8(void* p, size_t i, const float (&o)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) w[e] = f2h(o[2 * e]) | (f2h(o[2 * e + 1]) << 16);
    *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p) + i) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};
template <> struct ElemCodec<2> {                    // fp16
  __device__ static float h2f(uint32_t u) { const uint16_t s = (uint16_t)u; return __half2float(*reinterpret_cast<const __half*>(&s)); }
  __device__ static uint32_t f2h(float x) { __half h = __float2half_rn(x); return *reinterpret_cast<uint16_t*>(&h); }
  __device__ static float load(const void* p, size_t i) { return h2f(__ldg(reinterpret_cast<const uint16_t*>(p) + i)); }
  __device__ static void load8(const void* p, size_t i, float (&f)[8]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p) + i));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) { f[2 * e] = h2f(w[e] & 0xffffu); f[2 * e + 1] = h2f(w[e] >> 16); }
  }
  __device__ static void store(void* p, size_t i, float v) { reinterpret_cast<uint16_t*>(p)[i] = (uint16_t)f2h(v); }
  __device__ static void store8(void* p, size_t i, const float (&o)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) w[e] = f2h(o[2 * e]) | (f2h(o[2 * e + 1]) << 16);
    *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p) + i) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};
