// Callers on the wire side of the ML-KEM core (SURVEY.md 8(f) row 4), batched on the device:
//   dh/x25519/key.go:44-56                      KeyGen / Shared            -> x25519_kernel (thread per op)
//   kem/xwing/xwing.go:47-66,108-130,209-272    X-Wing                      -> expand / combiner kernels around the
//   kem/hybrid/hybrid.go:197-283, xkem.go       X25519MLKEM768,                ML-KEM / Kyber flows of mlkem.cu
//                                               Kyber768-X25519, Kyber512-X25519
// The lattice half of every scheme runs through the same device flows as cb200_mlkem_* / cb200_kyber_kem_*
// (mlkem_internal.h); this file adds the curve half, the SHAKE256 seed splitting, the X-Wing combiner and the
// strided copies that put the two halves next to each other in the packed keys and ciphertexts.
#include <algorithm>
#include <cstring>
#include <initializer_list>

#include "../../include/circl_b200.h"
#include "context.h"
#include "keccak.cuh"
#include "mlkem_internal.h"
#include "x25519.cuh"

namespace cb200 {
namespace hybrid {

__device__ __forceinline__ void ld8(uint32_t (&w)[8], const uint8_t* p) {
#pragma unroll
  for (int i = 0; i < 8; i++) w[i] = reinterpret_cast<const uint32_t*>(p)[i];
}
__device__ __forceinline__ void st8(uint8_t* p, const uint32_t (&w)[8]) {
#pragma unroll
  for (int i = 0; i < 8; i++) reinterpret_cast<uint32_t*>(p)[i] = w[i];
}

// out[i] = X25519(scalar[i], point[i] or the base point); status[i] |= 1 when the point is of small order
// (x25519.Shared returning false -> kem.ErrPubKey in xkem.go:150-152).  All strides are multiples of 4.
__global__ void __launch_bounds__(128, 2) x25519_kernel(const uint8_t* __restrict__ scalars, size_t s_stride,
                                                     const uint8_t* __restrict__ points, size_t p_stride,
                                                     uint8_t* __restrict__ out, size_t o_stride, uint8_t* __restrict__ status,
                                                     size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t k[8], p[8], r[8];
  ld8(k, scalars + i * s_stride);
  if (points) {
    ld8(p, points + i * p_stride);
  } else {
    p[0] = 9;
#pragma unroll
    for (int q = 1; q < 8; q++) p[q] = 0;
  }
  const bool ok = x25519::scalarmult(r, k, p);
  st8(out + i * o_stride, r);
  if (status && !ok) status[i] |= 1;
}

// out[i] = X25519(scalar[i], base point) through the fixed-base table (x25519.cuh): x25519.KeyGen (key.go:44-46)
__global__ void __launch_bounds__(128) x25519_base_kernel(const uint8_t* __restrict__ scalars, size_t s_stride,
                                                          uint8_t* __restrict__ out, size_t o_stride,
                                                          const int32_t* __restrict__ table, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t k[8], r[8];
  ld8(k, scalars + i * s_stride);
  x25519::scalarmult_base(r, k, table);
  st8(out + i * o_stride, r);
}

// out[i] = SHAKE256(in[i] (inlen bytes, <= 64), outlen <= 128 bytes), thread per op; inlen and outlen multiples of 8
__global__ void __launch_bounds__(128) shake_kernel(const uint8_t* __restrict__ in, size_t in_stride, int inlen,
                                                    uint8_t* __restrict__ out, size_t out_stride, int outlen, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t a[25];
  keccak::zero(a);
  const uint32_t* src = reinterpret_cast<const uint32_t*>(in + i * in_stride);
#pragma unroll
  for (int w = 0; w < 8; w++)
    if (8 * w < inlen) a[w] = (uint64_t)src[2 * w] | ((uint64_t)src[2 * w + 1] << 32);
  a[inlen / 8] ^= 0x1f;
  a[16] ^= 0x8000000000000000ull;
  keccak::f1600(a);
  uint32_t* dst = reinterpret_cast<uint32_t*>(out + i * out_stride);
#pragma unroll
  for (int w = 0; w < 16; w++)
    if (8 * w < outlen) {
      dst[2 * w] = (uint32_t)a[w];
      dst[2 * w + 1] = (uint32_t)(a[w] >> 32);
    }
}

// ss = SHA3-256(ss_M || ss_X || ct_X || pk_X || "\.//^\")  (xwing.go:47-66): 134 bytes, one block
__global__ void __launch_bounds__(128) xwing_combiner_kernel(const uint8_t* __restrict__ ssm, const uint8_t* __restrict__ ssx,
                                                             const uint8_t* __restrict__ ctx, size_t ctx_stride,
                                                             const uint8_t* __restrict__ pkx, size_t pkx_stride,
                                                             uint8_t* __restrict__ ss, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t a[25];
  keccak::zero(a);
  const uint32_t* src[4] = {reinterpret_cast<const uint32_t*>(ssm + 32 * i), reinterpret_cast<const uint32_t*>(ssx + 32 * i),
                            reinterpret_cast<const uint32_t*>(ctx + i * ctx_stride),
                            reinterpret_cast<const uint32_t*>(pkx + i * pkx_stride)};
#pragma unroll
  for (int s = 0; s < 4; s++)
#pragma unroll
    for (int w = 0; w < 4; w++) a[4 * s + w] = (uint64_t)src[s][2 * w] | ((uint64_t)src[s][2 * w + 1] << 32);
  // label 5c 2e 2f 2f 5e 5c, then the SHA-3 suffix 06 at byte 134 and 80 at byte 135
  a[16] = 0x5cull | (0x2eull << 8) | (0x2full << 16) | (0x2full << 24) | (0x5eull << 32) | (0x5cull << 40) | (0x06ull << 48) |
          (0x80ull << 56);
  keccak::f1600(a);
#pragma unroll
  for (int w = 0; w < 4; w++) {
    reinterpret_cast<uint32_t*>(ss + 32 * i)[2 * w] = (uint32_t)a[w];
    reinterpret_cast<uint32_t*>(ss + 32 * i)[2 * w + 1] = (uint32_t)(a[w] >> 32);
  }
}

// dst[i][0..width) = src[i][0..width): rows of 16-byte units between buffers of different strides
__global__ void __launch_bounds__(256) copy_rows_kernel(const uint8_t* __restrict__ src, size_t src_stride,
                                                        uint8_t* __restrict__ dst, size_t dst_stride, int units, size_t n) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * units) return;
  const size_t i = t / units;
  const int u = (int)(t % units);
  reinterpret_cast<uint4*>(dst + i * dst_stride)[u] = reinterpret_cast<const uint4*>(src + i * src_stride)[u];
}
__global__ void or_status_kernel(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint8_t mask, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && src[i]) dst[i] |= mask;
}

// ------------------------------------------------------------------ host side
static inline unsigned blocks(size_t units, size_t per) { return (unsigned)((units + per - 1) / per); }
static void copy_rows(const uint8_t* src, size_t ss, uint8_t* dst, size_t ds, size_t width, size_t n, cudaStream_t st) {
  KernelScope ks(KID_HYBRID_GLUE, st);
  copy_rows_kernel<<<blocks(n * (width / 16), 256), 256, 0, st>>>(src, ss, dst, ds, (int)(width / 16), n);
}
static void x25519_launch(const uint8_t* k, size_t ks_, const uint8_t* p, size_t ps, uint8_t* o, size_t os, uint8_t* status,
                          size_t n, cudaStream_t st) {
  KernelScope ks(KID_X25519, st);
  if (p)
    x25519_kernel<<<blocks(n, 128), 128, 0, st>>>(k, ks_, p, ps, o, os, status, n);
  else  // KeyGen: the base point never has small order, status stays untouched
    x25519_base_kernel<<<blocks(n, 128), 128, 0, st>>>(k, ks_, o, os, (const int32_t*)ctx().x25519_table, n);
}
static void shake_launch(const uint8_t* in, size_t is, int inlen, uint8_t* out, size_t os, int outlen, size_t n,
                         cudaStream_t st) {
  KernelScope ks(KID_HYBRID_GLUE, st);
  shake_kernel<<<blocks(n, 128), 128, 0, st>>>(in, is, inlen, out, os, outlen, n);
}

struct Arena {  // bump allocator over the second-level work area of a slot
  char* base = nullptr;
  size_t off = 0;
  uint8_t* take(size_t bytes) {
    uint8_t* p = (uint8_t*)(base + off);
    off += (bytes + 255) & ~(size_t)255;
    return p;
  }
};
static int arena(int slot, size_t bytes, Arena* a) {
  void* p = nullptr;
  int rc = ensure_work(kLevel1 + slot, bytes + 4096, &p);  // the level-1 areas belong to this file, level 0 to the lattice flows
  if (rc) return rc;
  a->base = (char*)p;
  a->off = 0;
  return 0;
}

// ---- X-Wing (ML-KEM-768 + X25519): pk = ek || pk_X (1216), sk = seed (32), ct = ct_M || ct_X (1120)
static int xwing_expand(const uint8_t* seeds, size_t stride, Arena& A, size_t n, cudaStream_t st, int slot, uint8_t** ek,
                        uint8_t** dk, uint8_t** ex) {
  *ex = A.take(n * 96);  // SHAKE256(seed, 96) = ML-KEM seed d || z (64) | X25519 secret (32)   (xwing.go:118-123)
  uint8_t* ms = A.take(n * 64);
  *ek = A.take(n * 1184);
  *dk = A.take(n * 2400);
  shake_launch(seeds, stride, 32, *ex, 96, 96, n, st);
  copy_rows(*ex, 96, ms, 64, 64, n, st);
  return mlkem::dev_keygen(3, 1, ms, *ek, *dk, n, st, slot);
}
static int xwing_keygen_dev(const uint8_t* seeds, uint8_t* pk, size_t n, cudaStream_t st, int slot) {
  Arena A;
  int rc = arena(slot, n * (96 + 64 + 1184 + 2400) + 4096, &A);
  if (rc) return rc;
  uint8_t *ek, *dk, *ex;
  rc = xwing_expand(seeds, 32, A, n, st, slot, &ek, &dk, &ex);
  if (rc) return rc;
  copy_rows(ek, 1184, pk, 1216, 1184, n, st);
  x25519_launch(ex + 64, 96, nullptr, 0, pk + 1184, 1216, nullptr, n, st);
  CB200_CUDA(cudaGetLastError());
  return 0;
}
static int xwing_encaps_dev(const uint8_t* pk, size_t pk_stride, const uint8_t* eseed, uint8_t* ct, uint8_t* ss,
                            uint8_t* status, size_t n, cudaStream_t st, int slot) {
  Arena A;
  int rc = arena(slot, n * (32 + 1088 + 32 + 32) + 4096, &A);
  if (rc) return rc;
  uint8_t *m = A.take(n * 32), *ctm = A.take(n * 1088), *ssm = A.take(n * 32), *ssx = A.take(n * 32);
  copy_rows(eseed, 64, m, 32, 32, n, st);
  rc = mlkem::dev_encaps(3, 1, pk, pk_stride, m, ctm, ssm, status, n, st, slot);
  if (rc) return rc;
  copy_rows(ctm, 1088, ct, 1120, 1088, n, st);
  x25519_launch(eseed + 32, 64, nullptr, 0, ct + 1088, 1120, nullptr, n, st);            // ct_X = KeyGen(ek_X)
  x25519_launch(eseed + 32, 64, pk + 1184, pk_stride, ssx, 32, nullptr, n, st);           // ss_X = Shared(ek_X, pk_X)
  {
    KernelScope ks(KID_HYBRID_GLUE, st);
    xwing_combiner_kernel<<<blocks(n, 128), 128, 0, st>>>(ssm, ssx, ct + 1088, 1120, pk + 1184, pk_stride, ss, n);
  }
  CB200_CUDA(cudaGetLastError());
  return 0;
}
static int xwing_decaps_dev(const uint8_t* sk, size_t sk_stride, const uint8_t* ct, uint8_t* ss, size_t n, cudaStream_t st,
                            int slot) {
  Arena A;
  int rc = arena(slot, n * (96 + 64 + 1184 + 2400 + 1088 + 32 + 32 + 32) + 8192, &A);
  if (rc) return rc;
  uint8_t *ek, *dk, *ex;
  rc = xwing_expand(sk, sk_stride, A, n, st, slot, &ek, &dk, &ex);  // sk.Unpack = deriveKeyPair (xwing.go:278-281)
  if (rc) return rc;
  uint8_t *ctm = A.take(n * 1088), *ssm = A.take(n * 32), *ssx = A.take(n * 32), *pkx = A.take(n * 32);
  copy_rows(ct, 1120, ctm, 1088, 1088, n, st);
  rc = mlkem::dev_decaps(3, 1, dk, 2400, ctm, ssm, nullptr, n, st, slot);
  if (rc) return rc;
  x25519_launch(ex + 64, 96, nullptr, 0, pkx, 32, nullptr, n, st);
  x25519_launch(ex + 64, 96, ct + 1088, 1120, ssx, 32, nullptr, n, st);
  {
    KernelScope ks(KID_HYBRID_GLUE, st);
    xwing_combiner_kernel<<<blocks(n, 128), 128, 0, st>>>(ssm, ssx, ct + 1088, 1120, pkx, 32, ss, n);
  }
  CB200_CUDA(cudaGetLastError());
  return 0;
}

// ---- kem/hybrid: two KEMs side by side (hybrid.go:197-283); the X25519 "KEM" is xkem.go
struct Hyb {
  int k, mlkem, x_first;
  size_t ek, dk, ct;  // sizes of the lattice half
};
static bool hyb_of(int id, Hyb* h) {
  switch (id) {
    case CB200_HYBRID_X25519MLKEM768: *h = {3, 1, 0, 1184, 2400, 1088}; return true;  // hybrid.go:58-62
    case CB200_HYBRID_KYBER768_X25519: *h = {3, 0, 1, 1184, 2400, 1088}; return true;  // hybrid.go:40-44
    case CB200_HYBRID_KYBER512_X25519: *h = {2, 0, 1, 800, 1632, 768}; return true;    // hybrid.go:34-38
  }
  return false;
}
static int hybrid_keygen_dev(const Hyb& H, const uint8_t* seeds, uint8_t* pk, uint8_t* sk, size_t n, cudaStream_t st,
                             int slot) {
  Arena A;
  int rc = arena(slot, n * (96 + 64 + 32 + H.ek + H.dk) + 8192, &A);
  if (rc) return rc;
  uint8_t *ex = A.take(n * 96), *ms = A.take(n * 64), *ek = A.take(n * H.ek), *dk = A.take(n * H.dk);
  const size_t pks = H.ek + 32, sks = H.dk + 32;
  const size_t xo_seed = H.x_first ? 0 : 64, mo_seed = H.x_first ? 32 : 0;  // hybrid.go:201-206
  uint8_t *pkx = pk + (H.x_first ? 0 : H.ek), *pkm = pk + (H.x_first ? 32 : 0);
  uint8_t *skx = sk + (H.x_first ? 0 : H.dk), *skm = sk + (H.x_first ? 32 : 0);
  shake_launch(seeds, 64, 64, ex, 96, 96, n, st);
  shake_launch(ex + xo_seed, 96, 32, skx, sks, 32, n, st);  // xkem.go:118-129: sk = SHAKE256(seed, 32)
  x25519_launch(skx, sks, nullptr, 0, pkx, pks, nullptr, n, st);
  copy_rows(ex + mo_seed, 96, ms, 64, 64, n, st);
  rc = mlkem::dev_keygen(H.k, H.mlkem, ms, ek, dk, n, st, slot);
  if (rc) return rc;
  copy_rows(ek, H.ek, pkm, pks, H.ek, n, st);
  copy_rows(dk, H.dk, skm, sks, H.dk, n, st);
  CB200_CUDA(cudaGetLastError());
  return 0;
}
static int hybrid_encaps_dev(const Hyb& H, const uint8_t* pk, size_t pk_stride, const uint8_t* seeds, uint8_t* ct,
                             uint8_t* ss, uint8_t* status, size_t n, cudaStream_t st, int slot) {
  Arena A;
  int rc = arena(slot, n * (64 + 32 + 32 + H.ct + 32 + 1) + 8192, &A);
  if (rc) return rc;
  uint8_t *ex = A.take(n * 64), *m = A.take(n * 32), *esk = A.take(n * 32), *ctm = A.take(n * H.ct), *ssm = A.take(n * 32),
          *st_m = A.take(n);
  const size_t cts = H.ct + 32;
  const size_t xo = H.x_first ? 0 : 32, mo = H.x_first ? 32 : 0;  // hybrid.go:240-245
  const uint8_t *pkx = pk + (H.x_first ? 0 : H.ek), *pkm = pk + (H.x_first ? 32 : 0);
  uint8_t *ctx = ct + (H.x_first ? 0 : H.ct), *ctmo = ct + (H.x_first ? 32 : 0);
  CB200_CUDA(cudaMemsetAsync(status, 0, n, st));
  CB200_CUDA(cudaMemsetAsync(st_m, 0, n, st));
  shake_launch(seeds, 32, 32, ex, 64, 64, n, st);
  shake_launch(ex + xo, 64, 32, esk, 32, 32, n, st);              // ephemeral sk = SHAKE256(seed_X, 32)  (xkem.go:177)
  x25519_launch(esk, 32, nullptr, 0, ctx, cts, nullptr, n, st);   // ct_X = its public key
  x25519_launch(esk, 32, pkx, pk_stride, ss + xo, 64, status, n, st);
  copy_rows(ex + mo, 64, m, 32, 32, n, st);
  rc = mlkem::dev_encaps(H.k, H.mlkem, pkm, pk_stride, m, ctm, ssm, st_m, n, st, slot);
  if (rc) return rc;
  copy_rows(ctm, H.ct, ctmo, cts, H.ct, n, st);
  copy_rows(ssm, 32, ss + mo, 64, 32, n, st);
  {
    KernelScope ks(KID_HYBRID_GLUE, st);
    or_status_kernel<<<blocks(n, 256), 256, 0, st>>>(status, st_m, 1, n);
  }
  CB200_CUDA(cudaGetLastError());
  return 0;
}
// status bit 0: kem.ErrPubKey (small-order X25519 share), bit 1: kem.ErrPrivKey (ML-KEM H(ek) check)
static int hybrid_decaps_dev(const Hyb& H, const uint8_t* sk, size_t sk_stride, const uint8_t* ct, uint8_t* ss,
                             uint8_t* status, size_t n, cudaStream_t st, int slot) {
  Arena A;
  int rc = arena(slot, n * (H.ct + 32 + 1) + 8192, &A);
  if (rc) return rc;
  uint8_t *ctm = A.take(n * H.ct), *ssm = A.take(n * 32), *st_m = A.take(n);
  const size_t cts = H.ct + 32;
  const size_t xo = H.x_first ? 0 : 32, mo = H.x_first ? 32 : 0;
  const uint8_t *skx = sk + (H.x_first ? 0 : H.dk), *skm = sk + (H.x_first ? 32 : 0);
  const uint8_t *ctx = ct + (H.x_first ? 0 : H.ct), *ctmi = ct + (H.x_first ? 32 : 0);
  CB200_CUDA(cudaMemsetAsync(status, 0, n, st));
  CB200_CUDA(cudaMemsetAsync(st_m, 0, n, st));
  x25519_launch(skx, sk_stride, ctx, cts, ss + xo, 64, status, n, st);
  copy_rows(ctmi, cts, ctm, H.ct, H.ct, n, st);
  rc = mlkem::dev_decaps(H.k, H.mlkem, skm, sk_stride, ctm, ssm, st_m, n, st, slot);
  if (rc) return rc;
  copy_rows(ssm, 32, ss + mo, 64, 32, n, st);
  {
    KernelScope ks(KID_HYBRID_GLUE, st);
    or_status_kernel<<<blocks(n, 256), 256, 0, st>>>(status, st_m, 2, n);
  }
  CB200_CUDA(cudaGetLastError());
  return 0;
}

// Every buffer of a call lives on the same side.  Host calls go through the staging pipeline in chunks.
static bool same_side(std::initializer_list<const void*> ps, bool* dev) {
  bool first = true;
  for (const void* p : ps) {
    if (!p) continue;
    const bool d = is_device_ptr(p);
    if (first) {
      *dev = d;
      first = false;
    } else if (d != *dev) {
      return false;
    }
  }
  return true;
}
// the first error class found among the per-op status bytes of a host-pointer call (counted by HostCall)
static int status_result(size_t pub, size_t priv, size_t n, const char* fn) {
  if (pub) {
    set_error("%s: %zu of %zu operations hit an invalid public key or key share (kem.ErrPubKey)", fn, pub, n);
    return CB200_ERR_PUBKEY;
  }
  if (priv) {
    set_error("%s: %zu of %zu decapsulation keys are inconsistent (kem.ErrPrivKey)", fn, priv, n);
    return CB200_ERR_PRIVKEY;
  }
  return 0;
}
// device-pointer calls read their buffers with 32-, 64- and 128-bit accesses
static bool aligned16(std::initializer_list<const void*> ps, std::initializer_list<size_t> strides) {
  uintptr_t acc = 0;
  for (const void* p : ps) acc |= (uintptr_t)p;
  for (size_t v : strides) acc |= v;
  return (acc & 15) == 0;
}

}  // namespace hybrid
}  // namespace cb200

using namespace cb200;
using namespace cb200::hybrid;

extern "C" {

int cb200_x25519(const uint8_t* scalars, const uint8_t* points, uint8_t* out, uint8_t* status, size_t n) {
  int rc = require_ready();
  if (rc) return rc;
  if (!scalars || !out) {
    set_error("cb200_x25519: null pointer");
    return CB200_ERR_ARG;
  }
  if (n == 0) return 0;
  bool dev = false;
  if (!same_side({scalars, points, out, status}, &dev)) {
    set_error("cb200_x25519: mixed host/device pointers");
    return CB200_ERR_ARG;
  }
  if (dev) {
    if (!aligned16({scalars, points, out}, {})) {
      set_error("cb200_x25519: device buffers must be 16-byte aligned");
      return CB200_ERR_ARG;
    }
    DeviceCall call(out);
    if (call.rc) return call.rc;
    if (status) CB200_CUDA(cudaMemsetAsync(status, 0, n, call.st));
    x25519_launch(scalars, 32, points, 32, out, 32, status, n, call.st);
    CB200_CUDA(cudaGetLastError());
    return 0;
  }
  HostCall hc;
  hc.bufs = {Buf{scalars, nullptr, 32, false, 0}, Buf{nullptr, out, 32, false, 0}, Buf{nullptr, nullptr, 1, false, 0}};
  if (points) hc.bufs.push_back(Buf{points, nullptr, 32, false, 0});
  hc.chunk = 1u << 17;
  hc.min_shard = 1u << 14;
  hc.status_buf = 2;
  hc.user_status = status;
  hc.body = [&](void** d, size_t cnt, size_t, cudaStream_t st, int) -> int {
    CB200_CUDA(cudaMemsetAsync(d[2], 0, cnt, st));
    x25519_launch((const uint8_t*)d[0], 32, points ? (const uint8_t*)d[3] : nullptr, 32, (uint8_t*)d[1], 32, (uint8_t*)d[2],
                  cnt, st);
    CB200_CUDA(cudaGetLastError());
    return 0;
  };
  rc = hc.run(n);
  if (rc) return rc;
  return status_result(hc.bit0, hc.bit1, n, "cb200_x25519");
}

int cb200_xwing_keygen(const uint8_t* seeds, uint8_t* pk, size_t n) {
  int rc = require_ready();
  if (rc) return rc;
  if (!seeds || !pk) {
    set_error("cb200_xwing_keygen: null pointer");
    return CB200_ERR_ARG;
  }
  if (n == 0) return 0;
  bool dev = false;
  if (!same_side({seeds, pk}, &dev)) {
    set_error("cb200_xwing_keygen: mixed host/device pointers");
    return CB200_ERR_ARG;
  }
  if (dev) {
    if (!aligned16({seeds, pk}, {})) {
      set_error("cb200_xwing_keygen: device buffers must be 16-byte aligned");
      return CB200_ERR_ARG;
    }
    DeviceCall call(pk);
    if (call.rc) return call.rc;
    return xwing_keygen_dev(seeds, pk, n, call.st, kDevSlot);
  }
  std::vector<Buf> bufs = {Buf{seeds, nullptr, 32, false, 0}, Buf{nullptr, pk, 1216, false, 0}};
  return run_host(bufs, n, 1u << 15, 1u << 13, [&](void** d, size_t cnt, size_t, cudaStream_t st, int slot) {
    return xwing_keygen_dev((const uint8_t*)d[0], (uint8_t*)d[1], cnt, st, slot);
  });
}

int cb200_xwing_encaps(const uint8_t* pk, size_t pk_stride, const uint8_t* eseeds, uint8_t* ct, uint8_t* ss, uint8_t* status,
                       size_t n) {
  int rc = require_ready();
  if (rc) return rc;
  if (!pk || !eseeds || !ct || !ss || (pk_stride != 0 && pk_stride < 1216)) {
    set_error("cb200_xwing_encaps: bad argument");
    return CB200_ERR_ARG;
  }
  if (n == 0) return 0;
  bool dev = false;
  if (!same_side({pk, eseeds, ct, ss, status}, &dev)) {
    set_error("cb200_xwing_encaps: mixed host/device pointers");
    return CB200_ERR_ARG;
  }
  if (dev) {
    if (!aligned16({pk, eseeds, ct, ss}, {pk_stride})) {
      set_error("cb200_xwing_encaps: device buffers and pk_stride must be 16-byte aligned");
      return CB200_ERR_ARG;
    }
    DeviceCall call(ct);
    if (call.rc) return call.rc;
    return xwing_encaps_dev(pk, pk_stride, eseeds, ct, ss, status, n, call.st, kDevSlot);
  }
  HostCall hc;
  hc.bufs = {Buf{pk, nullptr, 1216, pk_stride == 0, pk_stride}, Buf{eseeds, nullptr, 64, false, 0},
             Buf{nullptr, ct, 1120, false, 0}, Buf{nullptr, ss, 32, false, 0}, Buf{nullptr, nullptr, 1, false, 0}};
  hc.chunk = 1u << 15;
  hc.min_shard = 1u << 13;
  hc.status_buf = 4;
  hc.user_status = status;
  hc.body = [&](void** d, size_t cnt, size_t, cudaStream_t st, int slot) {
    return xwing_encaps_dev((const uint8_t*)d[0], pk_stride == 0 ? 0 : 1216, (const uint8_t*)d[1], (uint8_t*)d[2],
                            (uint8_t*)d[3], (uint8_t*)d[4], cnt, st, slot);
  };
  rc = hc.run(n);
  if (rc) return rc;
  return status_result(hc.bit0, hc.bit1, n, "cb200_xwing_encaps");
}

int cb200_xwing_decaps(const uint8_t* sk, size_t sk_stride, const uint8_t* ct, uint8_t* ss, size_t n) {
  int rc = require_ready();
  if (rc) return rc;
  if (!sk || !ct || !ss || (sk_stride != 0 && sk_stride < 32)) {
    set_error("cb200_xwing_decaps: bad argument");
    return CB200_ERR_ARG;
  }
  if (n == 0) return 0;
  bool dev = false;
  if (!same_side({sk, ct, ss}, &dev)) {
    set_error("cb200_xwing_decaps: mixed host/device pointers");
    return CB200_ERR_ARG;
  }
  if (dev) {
    if (!aligned16({sk, ct, ss}, {sk_stride})) {
      set_error("cb200_xwing_decaps: device buffers and sk_stride must be 16-byte aligned");
      return CB200_ERR_ARG;
    }
    DeviceCall call(ss);
    if (call.rc) return call.rc;
    return xwing_decaps_dev(sk, sk_stride, ct, ss, n, call.st, kDevSlot);
  }
  std::vector<Buf> bufs = {Buf{sk, nullptr, 32, sk_stride == 0, sk_stride}, Buf{ct, nullptr, 1120, false, 0},
                           Buf{nullptr, ss, 32, false, 0}};
  return run_host(bufs, n, 1u << 15, 1u << 13, [&](void** d, size_t cnt, size_t, cudaStream_t st, int slot) {
    return xwing_decaps_dev((const uint8_t*)d[0], sk_stride == 0 ? 0 : 32, (const uint8_t*)d[1], (uint8_t*)d[2], cnt, st, slot);
  });
}

size_t cb200_hybrid_public_key_size(int id) {
  Hyb h;
  return hyb_of(id, &h) ? h.ek + 32 : 0;
}
size_t cb200_hybrid_private_key_size(int id) {
  Hyb h;
  return hyb_of(id, &h) ? h.dk + 32 : 0;
}
size_t cb200_hybrid_ciphertext_size(int id) {
  Hyb h;
  return hyb_of(id, &h) ? h.ct + 32 : 0;
}

int cb200_hybrid_keygen(int id, const uint8_t* seeds, uint8_t* pk, uint8_t* sk, size_t n) {
  int rc = require_ready();
  if (rc) return rc;
  Hyb H;
  if (!hyb_of(id, &H) || !seeds || !pk || !sk) {
    set_error("cb200_hybrid_keygen: bad argument");
    return CB200_ERR_ARG;
  }
  if (n == 0) return 0;
  bool dev = false;
  if (!same_side({seeds, pk, sk}, &dev)) {
    set_error("cb200_hybrid_keygen: mixed host/device pointers");
    return CB200_ERR_ARG;
  }
  if (dev) {
    if (!aligned16({seeds, pk, sk}, {})) {
      set_error("cb200_hybrid_keygen: device buffers must be 16-byte aligned");
      return CB200_ERR_ARG;
    }
    DeviceCall call(pk);
    if (call.rc) return call.rc;
    return hybrid_keygen_dev(H, seeds, pk, sk, n, call.st, kDevSlot);
  }
  std::vector<Buf> bufs = {Buf{seeds, nullptr, 64, false, 0}, Buf{nullptr, pk, H.ek + 32, false, 0},
                           Buf{nullptr, sk, H.dk + 32, false, 0}};
  return run_host(bufs, n, 1u << 15, 1u << 13, [&](void** d, size_t cnt, size_t, cudaStream_t st, int slot) {
    return hybrid_keygen_dev(H, (const uint8_t*)d[0], (uint8_t*)d[1], (uint8_t*)d[2], cnt, st, slot);
  });
}

int cb200_hybrid_encaps(int id, const uint8_t* pk, size_t pk_stride, const uint8_t* seeds, uint8_t* ct, uint8_t* ss,
                        uint8_t* status, size_t n) {
  int rc = require_ready();
  if (rc) return rc;
  Hyb H;
  if (!hyb_of(id, &H) || !pk || !seeds || !ct || !ss || (pk_stride != 0 && pk_stride < H.ek + 32)) {
    set_error("cb200_hybrid_encaps: bad argument");
    return CB200_ERR_ARG;
  }
  if (n == 0) return 0;
  bool dev = false;
  if (!same_side({pk, seeds, ct, ss, status}, &dev)) {
    set_error("cb200_hybrid_encaps: mixed host/device pointers");
    return CB200_ERR_ARG;
  }
  if (dev) {
    if (!status) {
      set_error("cb200_hybrid_encaps: device-pointer calls need a status array (it carries kem.ErrPubKey)");
      return CB200_ERR_ARG;
    }
    if (!aligned16({pk, seeds, ct, ss}, {pk_stride})) {
      set_error("cb200_hybrid_encaps: device buffers and pk_stride must be 16-byte aligned");
      return CB200_ERR_ARG;
    }
    DeviceCall call(ct);
    if (call.rc) return call.rc;
    return hybrid_encaps_dev(H, pk, pk_stride, seeds, ct, ss, status, n, call.st, kDevSlot);
  }
  const size_t pks = H.ek + 32;
  HostCall hc;
  hc.bufs = {Buf{pk, nullptr, pks, pk_stride == 0, pk_stride}, Buf{seeds, nullptr, 32, false, 0},
             Buf{nullptr, ct, H.ct + 32, false, 0}, Buf{nullptr, ss, 64, false, 0}, Buf{nullptr, nullptr, 1, false, 0}};
  hc.chunk = 1u << 15;
  hc.min_shard = 1u << 13;
  hc.status_buf = 4;
  hc.user_status = status;
  hc.body = [&](void** d, size_t cnt, size_t, cudaStream_t st, int slot) {
    return hybrid_encaps_dev(H, (const uint8_t*)d[0], pk_stride == 0 ? 0 : pks, (const uint8_t*)d[1], (uint8_t*)d[2],
                             (uint8_t*)d[3], (uint8_t*)d[4], cnt, st, slot);
  };
  rc = hc.run(n);
  if (rc) return rc;
  return status_result(hc.bit0, hc.bit1, n, "cb200_hybrid_encaps");
}

int cb200_hybrid_decaps(int id, const uint8_t* sk, size_t sk_stride, const uint8_t* ct, uint8_t* ss, uint8_t* status, size_t n) {
  int rc = require_ready();
  if (rc) return rc;
  Hyb H;
  if (!hyb_of(id, &H) || !sk || !ct || !ss || sk_stride < H.dk + 32) {
    set_error("cb200_hybrid_decaps: bad argument (one decapsulation key per operation: sk_stride >= key size)");
    return CB200_ERR_ARG;
  }
  if (n == 0) return 0;
  bool dev = false;
  if (!same_side({sk, ct, ss, status}, &dev)) {
    set_error("cb200_hybrid_decaps: mixed host/device pointers");
    return CB200_ERR_ARG;
  }
  if (dev) {
    if (!status) {
      set_error("cb200_hybrid_decaps: device-pointer calls need a status array (it carries kem.ErrPubKey / kem.ErrPrivKey)");
      return CB200_ERR_ARG;
    }
    if (!aligned16({sk, ct, ss}, {sk_stride})) {
      set_error("cb200_hybrid_decaps: device buffers and sk_stride must be 16-byte aligned");
      return CB200_ERR_ARG;
    }
    DeviceCall call(ss);
    if (call.rc) return call.rc;
    return hybrid_decaps_dev(H, sk, sk_stride, ct, ss, status, n, call.st, kDevSlot);
  }
  const size_t sks = H.dk + 32;
  HostCall hc;
  hc.bufs = {Buf{sk, nullptr, sks, false, sk_stride}, Buf{ct, nullptr, H.ct + 32, false, 0},
             Buf{nullptr, ss, 64, false, 0}, Buf{nullptr, nullptr, 1, false, 0}};
  hc.chunk = 1u << 15;
  hc.min_shard = 1u << 13;
  hc.status_buf = 3;
  hc.user_status = status;
  hc.body = [&](void** d, size_t cnt, size_t, cudaStream_t st, int slot) {
    return hybrid_decaps_dev(H, (const uint8_t*)d[0], sks, (const uint8_t*)d[1], (uint8_t*)d[2], (uint8_t*)d[3], cnt, st, slot);
  };
  rc = hc.run(n);
  if (rc) return rc;
  return status_result(hc.bit0, hc.bit1, n, "cb200_hybrid_decaps");
}

}  // extern "C"
