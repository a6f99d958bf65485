// sph_common.cuh — shared device/host definitions of the B200 SPH step engine.
//
// Data layout in HBM (all FP64 SoA, particle arrays kept physically in the Morton order of the most
// recent evaluation; `id` carries the reference's `number`, SUMMER_SPH.f90:15,886-888):
//   state   : x y z vx vy vz u m alpha h            (10 x 8 B)  + id (4 B)     double-buffered for the re-order
//   derived : rho omega P c PoR2                    ( 5 x 8 B)
//   rates   : ax ay az udot alphadot                ( 5 x 8 B)
//   tree    : key (8 B) level (4 B) leaf centre cx cy cz (24 B) reach R = 2h + size/2 (8 B)
//   BVH     : per 32-particle chunk and per 8-ary group of chunks: position box + reach box, 12 floats
//   octree  : compressed Barnes-Hut octree in depth-first preorder, 48 B per node (COM, M, size, next)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#define SPH_KEY_LEVELS 21          // 3 bits per level in a 63-bit descent key word
#define SPH_KEY_LEVELS2 42         // two key words: levels 22..42 live in the second word (slow path)
#define SPH_CHUNK 32               // particles per BVH leaf chunk = one warp of targets
#define SPH_BVH_FAN 8
#define SPH_MAX_SINKS 64
#define FULL_MASK 0xffffffffu

#ifdef SCREEN_AUDIT    // developer build (scripts/build_variant.sh audit -DSCREEN_AUDIT): decisions of the FP32 screens that the FP64
                       // tests they stand in front of contradict: [0] density, [1] pair loop, [2] gravity (stderr per evaluation / step)
__device__ unsigned long long screen_audit[3];
#endif

struct DevParams {
  int    variable_h;     // V mode
  int    soft_hi;        // T:298 softening
  int    nq;
  int    lmax;           // min(max_depth, levels the key can hold: 21, or 42 on the two-word slow path)
  int    depth_unbounded;// max_depth > lmax: particles sharing a full key are NOT a depth-limited leaf of the reference
  double dq, inv_dq;
  double h_fixed;
  double pi_norm;        // F:125 3.14159265359_dp | V:7 real(4) pi
  double gamma, gm1;
  double theta;
  double G;              // real(4) literal 39.478416442871094 (F:7)
  double eta, conv, max_length, tscale, bounding;
  double lit_001, lit_015, lit_01, lit_1em4;   // real(4) literals (SURVEY §8(a'))
};

// root cube of the current tree (device resident)
struct RootBox { double cx, cy, cz, size; double mn[3], mx[3]; };

// Barnes-Hut node, depth-first preorder; leaves are nodes too.
struct __align__(16) GNode {
  double cx, cy, cz, m;   // centre of mass, total mass
  double size;            // cell edge at the node's own (branching / leaf) level
  int    next;            // preorder index just past this node's subtree
  int    flags;           // bit0: childless (leaf or depth-limited multi-particle node)
};

// The same node in the gravity walk layout: children contiguous at [child, child + nchild); nchild == 0 for
// leaves and depth-limited childless nodes.
struct __align__(16) WNode {
  double cx, cy, cz, m;
  double size;
  int    child;
  int    nchild;
};

// float AABBs rounded outward; pos = particle positions, reach = union of leaf boxes expanded by 2h
struct __align__(16) BvhBox { float plo[3], phi[3], rlo[3], rhi[3]; };

__host__ __device__ inline uint64_t mix64(uint64_t z) {   // splitmix64 finaliser (same in oracle)
  z += 0x9E3779B97F4A7C15ull; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

#ifdef __CUDACC__
// number of leading octal digits (levels) two 63-bit keys share, capped at lmax
__device__ __forceinline__ int lcp_levels(uint64_t a, uint64_t b, int lmax) {
  uint64_t x = a ^ b;
  if (x == 0) return lmax;
  int l = (__clzll((long long)x) - 1) / 3;
  return l < lmax ? l : lmax;
}

// two-word keys: `lo` may be null (single-word fast path)
__device__ __forceinline__ int lcp_levels2(uint64_t ha, uint64_t la, uint64_t hb, uint64_t lb, int lmax) {
  uint64_t x = ha ^ hb;
  int l;
  if (x != 0) l = (__clzll((long long)x) - 1) / 3;
  else {
    uint64_t y = la ^ lb;
    if (y == 0) return lmax;
    l = SPH_KEY_LEVELS + (__clzll((long long)y) - 1) / 3;
  }
  return l < lmax ? l : lmax;
}
// octal digit of descent level l (0-based: l = 0 is the root's split)
__device__ __forceinline__ int key_digit(uint64_t hi, uint64_t lo, int l) {
  return l < SPH_KEY_LEVELS ? (int)((hi >> (3 * (SPH_KEY_LEVELS - 1 - l))) & 7)
                            : (int)((lo >> (3 * (SPH_KEY_LEVELS2 - 1 - l))) & 7);
}

// Reciprocal / square root without the IEEE slow-path subroutine: MUFU seed (~2^-20) + two FMA Newton /
// Goldschmidt steps (~1 ulp).  Used only where the result feeds FP64 sums compared at 1e-10; every
// membership / ordering decision uses the correctly rounded __d*_rn intrinsics instead.
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0); r = fma(r, e, r);
  e = fma(-x, r, 1.0); r = fma(r, e, r);
  return r;
}
// s = sqrt(x), rs = 1/sqrt(x) for x > 0 (x == 0 gives NaN in both, callers guard where 0 is legal)
__device__ __forceinline__ void fast_sqrt_rsqrt(double x, double& s, double& rs) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double g = x * y, h = 0.5 * y;
  double r = fma(-h, g, 0.5); g = fma(g, r, g); h = fma(h, r, h);
  r = fma(-h, g, 0.5); g = fma(g, r, g); h = fma(h, r, h);
  s = g; rs = 2.0 * h;
}

__device__ __forceinline__ double warp_min(double v) {
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL_MASK, v, o));
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL_MASK, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return v;
}
__device__ __forceinline__ float warp_minf(float v) {
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(FULL_MASK, v, o));
  return v;
}
__device__ __forceinline__ float warp_maxf(float v) {
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL_MASK, v, o));
  return v;
}
__device__ __forceinline__ long long warp_sum_ll(long long v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return v;
}
#endif
