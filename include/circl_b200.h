/*
 * include/circl_b200.h -- C ABI of libcirclb200.so, the B200 (sm_100a) batch
 * polynomial-ring engine behind CIRCL's module-lattice hot path.
 *
 * This is the surface a cgo shim binds (see INTEGRATION.md and go/).  Plain
 * pointers and sizes only.  Every buffer is caller-owned and never retained
 * past the call.  A pointer may be a host pointer (pageable or pinned) or a
 * CUDA device pointer; the library detects which (cudaPointerGetAttributes)
 * and stages host buffers through HBM itself.  Where a call takes a row stride
 * (op i uses base + i*stride), a host-pointer stride may be any value at least
 * the row size; device-pointer calls of the KEM and signature entry points
 * want their buffers and key strides 16-byte aligned (CB200_ERR_ARG
 * otherwise).  All entry points return 0 on
 * success or a negative code; cb200_last_error() gives the message.  There is
 * no CPU fallback: without a usable CUDA device every compute call fails.
 *
 * Citations are file:line in cloudflare/circl (the interface each entry point
 * replaces).  Coefficient order is the reference's standard ("detangled")
 * order; results are bit-identical to the reference's *Generic functions.
 */
#ifndef CIRCL_B200_H
#define CIRCL_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes (mapped by the Go shim to kem.Err*, kem/kem.go:92-121) ---- */
#define CB200_OK 0
#define CB200_ERR_ARG (-1)          /* programmer error: the Go shim panics, as the reference does */
#define CB200_ERR_NOT_INIT (-2)
#define CB200_ERR_PUBKEY (-3)       /* kem.ErrPubKey: ek not reduced mod q (cpapke.go:45-55); see cb200_mlkem_encaps */
#define CB200_ERR_SIGN_ATTEMPTS (-4)/* ML-DSA: 576 attempts exhausted (sign/mldsa/mldsa65/internal/dilithium.go:372-377) */
#define CB200_ERR_PRIVKEY (-5)      /* kem.ErrPrivKey: H(ek) inside dk does not match (kem/mlkem/mlkem768/kyber.go:226-228) */
/* <= -100: CUDA runtime error (-100 - cudaError_t) */

/* ---- lifetime ---- */
/* cb200_init_devices(ndev): one process drives GPUs 0..ndev-1 (ndev <= 0: every visible GPU).  Host-pointer batch
 * calls are then cut into one contiguous index range per GPU inside the library and the results land in the
 * caller's buffers in index order -- a kem.Scheme / sign.Scheme caller never sees devices (north_star: "batches
 * shard by index across the 8 GPUs").  cb200_init(device): exactly one GPU (the one-process-per-GPU launch).
 * Calling either again with another set re-initialises. */
int cb200_init(int device);
int cb200_init_devices(int ndev);
int cb200_active_devices(void);        /* GPUs this process was initialised on (0 = not initialised) */
void cb200_shutdown(void);
int cb200_device_count(void);
const char *cb200_last_error(void);    /* message of the last failing call on this thread */
const char *cb200_version(void);
/* Threading (kem/kem.go:33-82 and sign/sign.go:48-94 are goroutine-safe; so is this):
 *  - host-pointer calls may be issued from any number of threads; each GPU runs the ranges it is given one after
 *    the other on its own worker thread, small batches rotate over the GPUs;
 *  - device-pointer calls run on the GPU that owns the buffers, asynchronously on the CUDA stream (cudaStream_t cast
 *    to void*) the CALLING THREAD named with cb200_set_stream -- the setting is per thread; NULL, the initial state,
 *    is CUDA's legacy default stream.  Scratch memory is kept per (GPU, stream): calls on different streams never
 *    share it, calls on one stream from several threads are serialised in stream order.  cb200_release_stream frees
 *    the scratch of a stream that is about to be destroyed.  A cgo caller wraps set_stream + call in
 *    runtime.LockOSThread (go/cb200). */
int cb200_set_stream(void *cuda_stream);
int cb200_release_stream(void *cuda_stream);
int cb200_synchronize(void);           /* waits for this thread's stream */
/* Pins the calling thread to the CPUs next to GPU `device` (/sys/bus/pci/devices/<id>/local_cpulist); memory it
 * allocates and first touches afterwards is local to that GPU's NUMA node.  Returns the number of CPUs, 0 if the
 * topology is unknown (affinity unchanged).  The library's own worker threads do this themselves. */
int cb200_bind_thread_to_device(int device);
/* ---- result gather of the one-process-per-GPU launch (SURVEY.md 8(e)) ----
 * Rank 0 allocates the destination of the gather (plain cudaMalloc memory on its GPU) and gets a 64-byte handle to
 * publish over any transport (torch.distributed, a pipe); every other rank opens the handle and pushes its rows:
 * cb200_gather_push(dst, src, bytes) is a cudaMemcpyAsync into the mapped peer memory over NVLink, issued on a copy
 * stream of the library that first waits for everything the calling thread's stream has queued so far -- copy-engine
 * traffic, no SM, no NCCL kernel beside the compute kernels.  dst may also be local (rank 0's own rows).
 * cb200_gather_flush(row, wait_on_host): wait_on_host != 0 blocks until this rank's pushes have landed; otherwise the
 * calling thread's stream is made to wait for them.  `row` is any device pointer of the pushing GPU. */
#define CB200_GATHER_HANDLE_BYTES 64
int cb200_gather_alloc(size_t bytes, void **dev_ptr, uint8_t *handle);
int cb200_gather_free(void *dev_ptr);
int cb200_gather_open(const uint8_t *handle, void **peer_ptr);
int cb200_gather_close(void *peer_ptr);
int cb200_gather_push(void *dst, const void *src, size_t bytes);
int cb200_gather_flush(const void *any_local_row, int wait_on_host);
/* Pinned host memory for large batches handed to Go via unsafe.Slice. */
void *cb200_host_alloc(size_t bytes);
/* The same for one array of a batch (n rows of unit_bytes) that host-pointer calls will split over all active GPUs
 * (cb200_init_devices): the rows of each GPU's shard are placed on that GPU's NUMA node, so that all GPUs copy at link
 * speed at the same time instead of sharing the socket interconnect.  Freed with cb200_host_free. */
void *cb200_host_alloc_batch(size_t n, size_t unit_bytes);
void cb200_host_free(void *p);
/* number of kernels launched by this library since init (bench accounting) */
uint64_t cb200_launch_count(void);
/* Optional per-kernel-class timing with CUDA events on the launching stream
 * (used by bench.py for the roofline line).  cb200_profile_read synchronises the
 * device, fills ms_total[i] / launches[i] for the first n classes and clears. */
int cb200_profile_enable(int on);
int cb200_profile_kernel_count(void);
const char *cb200_profile_kernel_name(int id);
int cb200_profile_read(double *ms_total, uint64_t *launches, int n);

/* ---- Kyber / ML-KEM ring, q = 3329, Poly = [256]int16 ---- */
/* (*Poly).NTT / InvNTT   pke/kyber/internal/common/generic.go:24,36; stubs_amd64.go:8-14
 * in place over n contiguous polynomials.  Results equal nttGeneric / invNTTGeneric (ntt.go:60-193) bit for bit,
 * unnormalised, for EVERY int16 input (the reference's int16 wrap-around included).  Inputs inside the reference's
 * contract (|c| <= q; in fact |c| <= 13561 forward, <= 3679 inverse) run a faster kernel path. */
int cb200_kyber_ntt(int16_t *polys, size_t n, int inverse);
/* (*Poly).MulHat         generic.go:49; poly.go:63-100.  out may alias a or b. */
int cb200_kyber_mulhat(int16_t *out, const int16_t *a, const int16_t *b, size_t n);
/* PolyDotHat             pke/kyber/kyber768/internal/vec.go:30-37
 * a, b: n vectors of k polynomials; out: n polynomials. */
int cb200_kyber_dot(int16_t *out, const int16_t *a, const int16_t *b, int k, size_t n);
/* Add, Sub, BarrettReduce, Normalize, ToMont   generic.go:7-77, poly.go:13-52 */
#define CB200_OP_ADD 0
#define CB200_OP_SUB 1
#define CB200_OP_BARRETT 2
#define CB200_OP_NORMALIZE 3
#define CB200_OP_TOMONT 4
int cb200_kyber_poly_op(int op, int16_t *out, const int16_t *a, const int16_t *b, size_t n);

/* ---- Dilithium / ML-DSA ring, q = 8380417, Poly = [256]uint32 ---- */
/* (*Poly).NTT / InvNTT   sign/internal/dilithium/generic.go:11,15; stubs_amd64.go:8-14; in place */
int cb200_dil_ntt(uint32_t *polys, size_t n, int inverse);
/* (*Poly).MulHat         sign/internal/dilithium/generic.go:19 (poly.go:88) */
int cb200_dil_mulhat(uint32_t *out, const uint32_t *a, const uint32_t *b, size_t n);
/* PolyDotHat             sign/mldsa/mldsa65/internal/mat.go:52-59 (k = L polynomials per vector) */
int cb200_dil_dot(uint32_t *out, const uint32_t *a, const uint32_t *b, int k, size_t n);
/* Add, Sub, ReduceLe2Q, Normalize, NormalizeAssumingLe2Q, MulBy2toD   generic.go:23-89, poly.go:10-100 */
#define CB200_DIL_OP_ADD 0
#define CB200_DIL_OP_SUB 1
#define CB200_DIL_OP_REDUCE_LE2Q 2
#define CB200_DIL_OP_NORMALIZE 3
#define CB200_DIL_OP_NORMALIZE_LE2Q 4
#define CB200_DIL_OP_MUL_2D 5
int cb200_dil_poly_op(int op, uint32_t *out, const uint32_t *a, const uint32_t *b, size_t n);
/* (*Poly).Exceeds        poly.go:51-71 (stubs_amd64.go:32 exceedsAVX2): flags[i] = 1 iff poly i exceeds bound */
int cb200_dil_exceeds(const uint32_t *polys, uint32_t bound, uint8_t *flags, size_t n);

/* ---- Keccak (simd/keccakf1600, internal/sha3): the on-device sampler's permutation, batched ---- */
/* StateX4.Permute  simd/keccakf1600/f1600x.go:115-121 / KeccakF1600  internal/sha3/keccakf.go:12
 * states: n x 25 little-endian 64-bit lanes (200 bytes per state, lane x+5y at index x+5y), permuted in place;
 * turbo != 0: the 12-round TurboSHAKE variant (keccakf.go:12 `turbo`). */
int cb200_keccak_f1600(uint64_t *states, size_t n, int turbo);
/* One-shot sponges over n messages of equal length (internal/sha3/hashes.go:21,35; shake.go:56,74):
 * bits = 128 / 256 selects SHAKE128 / SHAKE256 with `outlen` output bytes, bits = -256 / -512 selects SHA3-256 /
 * SHA3-512 (outlen must be 32 / 64).  Message i = in + i*in_stride (in_stride 0: one message), output i at
 * out + i*outlen. */
int cb200_sha3(int bits, const uint8_t *in, size_t in_stride, size_t inlen, uint8_t *out, size_t outlen, size_t n);

/* ---- samplers of the Kyber ring (pke/kyber/internal/common/sample.go) ---- */
/* (*Poly).DeriveUniform  sample.go:192-236: polys[i] = 12-bit rejection sampling of SHAKE128(seed_i || x_i || y_i);
 * seeds: 32 bytes each at seeds + i*seed_stride (0: one seed); xy: n x 2 bytes (x, y). */
int cb200_kyber_derive_uniform(int16_t *polys, const uint8_t *seeds, size_t seed_stride, const uint8_t *xy, size_t n);
/* (*Poly).DeriveNoise(2|3)  sample.go:31-95: polys[i] = CBD_eta(SHAKE256(seed_i || nonce_i)); seeds 32 bytes each. */
int cb200_kyber_derive_noise(int16_t *polys, int eta, const uint8_t *seeds, size_t seed_stride, const uint8_t *nonces,
                             size_t n);
/* ---- serialisation of the Kyber ring (pke/kyber/internal/common/poly.go) ---- */
/* Pack / Unpack  poly.go:106-129: 12 bits per coefficient, 384 bytes per polynomial (input normalised) */
int cb200_kyber_pack(uint8_t *out, const int16_t *polys, size_t n);
int cb200_kyber_unpack(int16_t *polys, const uint8_t *in, size_t n);
/* CompressTo / Decompress  poly.go:170-328 for d in {4, 5, 10, 11} (32 d bytes per polynomial), and
 * CompressMessageTo / DecompressMessage  poly.go:134-166 for d = 1 (32 bytes); compress expects normalised input */
int cb200_kyber_compress(uint8_t *out, const int16_t *polys, int d, size_t n);
int cb200_kyber_decompress(int16_t *polys, const uint8_t *in, int d, size_t n);

/* ---- samplers and packers of the Dilithium ring; mode = 44, 65 or 87 picks the per-mode package
 *      (sign/mldsa/mldsa{44,65,87}/internal/sample.go, sign/internal/dilithium/generic.go) ---- */
/* PolyDeriveUniform  sample.go:92-123: 23-bit rejection sampling of SHAKE128(seed_i || le16(nonce_i)); seeds 32 bytes */
int cb200_dil_derive_uniform(uint32_t *polys, const uint8_t *seeds, size_t seed_stride, const uint16_t *nonces, size_t n);
/* PolyDeriveUniformLeqEta  sample.go:129-181: coefficients Q + eta - t, t from nibbles of SHAKE256(seed_i(64) || nonce) */
int cb200_dil_derive_leq_eta(int mode, uint32_t *polys, const uint8_t *seeds, size_t seed_stride, const uint16_t *nonces,
                             size_t n);
/* PolyDeriveUniformLeGamma1  sample.go:197-209: gamma1 - (18|20-bit fields of SHAKE256(seed_i(64) || nonce)), mod q */
int cb200_dil_derive_le_gamma1(int mode, uint32_t *polys, const uint8_t *seeds, size_t seed_stride,
                               const uint16_t *nonces, size_t n);
/* PolyDeriveUniformBall  sample.go:299-339: tau coefficients +-1 from SHAKE256(seed_i); seeds are c~ (32/48/64 bytes
 * for mode 44/65/87) at seeds + i*seed_stride */
int cb200_dil_derive_ball(int mode, uint32_t *polys, const uint8_t *seeds, size_t seed_stride, size_t n);
/* (*Poly).Power2Round  generic.go:85 (poly.go:77-84): a0plusq[i] = Q + a0, a1[i] for normalised a */
int cb200_dil_power2round(uint32_t *a0plusq, uint32_t *a1, const uint32_t *a, size_t n);
/* (*Poly).PackLe16  generic.go:27 (pack.go:102-108): 4 bits per coefficient, 128 bytes per polynomial */
int cb200_dil_pack_le16(uint8_t *out, const uint32_t *polys, size_t n);

/* ---- ML-KEM ---- */
/* scheme.UnmarshalBinaryPublicKey + EncapsulateDeterministically
 *   kem/mlkem/mlkem768/kyber.go:390-396,359-374,103-137 (mlkem1024: same lines)
 * k = 2 (ML-KEM-512: ek 800, ct 768), 3 (ML-KEM-768: ek 1184, ct 1088) or 4 (ML-KEM-1024: ek 1568, ct 1568).
 * ek_stride = 0: one ek shared by all n operations (parsed once);
 * otherwise op i uses ek + i*ek_stride and A^T, H(ek) are rebuilt on device per op.
 * seeds: n x 32 (the message m); ct: n x CiphertextSize; ss: n x 32.
 * status (optional, may be NULL): n bytes, 0 = ok, 1 = kem.ErrPubKey for that op
 * (its ct/ss are zeroed).  Returns CB200_ERR_PUBKEY if any op failed. */
int cb200_mlkem_encaps(int k, const uint8_t *ek, size_t ek_stride, const uint8_t *seeds, uint8_t *ct, uint8_t *ss,
                       uint8_t *status, size_t n);
/* The same on device pointers, with the result gather of the one-process-per-GPU launch fused into the flow: the rows of
 * every sub-batch (8192 operations) are also copied to push_ct + i*CiphertextSize / push_ss + i*32 -- typically this
 * rank's place in rank 0's cb200_gather_alloc buffer, opened with cb200_gather_open -- as soon as they exist, by the
 * copy engines over NVLink while the following sub-batches compute.  Either may be NULL.  The calling thread's stream
 * is ordered after the pushes. */
int cb200_mlkem_encaps_push(int k, const uint8_t *ek, size_t ek_stride, const uint8_t *seeds, uint8_t *ct, uint8_t *ss,
                            uint8_t *status, size_t n, uint8_t *push_ct, uint8_t *push_ss);
/* scheme.UnmarshalBinaryPrivateKey + Decapsulate
 *   kem/mlkem/mlkem768/kyber.go:398-407,376-388 -> PrivateKey.Unpack :203-229, DecapsulateTo :144-184
 *   (cpapke DecryptTo cpapke.go:113-130, re-encryption EncryptTo :137-181, implicit rejection with J = SHAKE256(z || ct)).
 * dk: packed decapsulation key(s) (2400 / 3168 bytes); op i uses dk + i*dk_stride (0 = one key, host pointers only).
 * ct: n x CiphertextSize; ss: n x 32.  status (optional): 2 = kem.ErrPrivKey for that op (ss zeroed).
 * Returns CB200_ERR_PRIVKEY if any op failed. */
int cb200_mlkem_decaps(int k, const uint8_t *dk, size_t dk_stride, const uint8_t *ct, uint8_t *ss, uint8_t *status,
                       size_t n);
/* scheme.DeriveKeyPair   kem/mlkem/mlkem768/kyber.go:337-346 -> NewKeyFromSeed :57-78 ->
 *   cpapke.NewKeyFromSeedMLKEM pke/kyber/kyber768/kyber.go:77-86 -> internal/cpapke.go:66-110.
 * seeds: n x 64 (d || z); ek: n x PublicKeySize; dk: n x PrivateKeySize (packed, = MarshalBinary). */
int cb200_mlkem_keygen(int k, const uint8_t *seeds, uint8_t *ek, uint8_t *dk, size_t n);
size_t cb200_mlkem_private_key_size(int k);
size_t cb200_mlkem_public_key_size(int k);
size_t cb200_mlkem_ciphertext_size(int k);

#define CB200_SIGN_INTERNAL 1 /* flags: ML-DSA.Sign_internal / Verify_internal on the message as given */

/* ---- round-3 Kyber512/768/1024 KEM (k = 2, 3, 4): kem/kyber/kyber768/kyber.go:56-198 ----
 * Same K-PKE and byte sizes as ML-KEM; the FO wrapper differs (m = H(seed), ss = KDF(K || H(ct)), key generation
 * without the K byte, no modulus check of ek, no H(ek) check of dk -- hence no status array).  Strides as in
 * cb200_mlkem_*: 0 = one key shared by all operations. */
int cb200_kyber_kem_keygen(int k, const uint8_t *seeds, uint8_t *ek, uint8_t *dk, size_t n);
int cb200_kyber_kem_encaps(int k, const uint8_t *ek, size_t ek_stride, const uint8_t *seeds, uint8_t *ct, uint8_t *ss,
                           size_t n);
int cb200_kyber_kem_decaps(int k, const uint8_t *dk, size_t dk_stride, const uint8_t *ct, uint8_t *ss, size_t n);

/* ---- callers on the wire side of ML-KEM (SURVEY.md 8(f) row 4) ----
 * cb200_x25519: dh/x25519 KeyGen (points == NULL: base point, key.go:44-46) or Shared (key.go:48-56) on n
 * 32-byte scalars / points; status[i] = 1 where the point has small order (Shared returning false); the output is
 * then all zero and the host-pointer call returns CB200_ERR_PUBKEY after finishing the batch. */
int cb200_x25519(const uint8_t *scalars, const uint8_t *points, uint8_t *out, uint8_t *status, size_t n);

/* X-Wing (kem/xwing/xwing.go:32-44): seed / sk 32, pk 1216 (ML-KEM-768 ek || X25519 pk), encapsulation seed 64,
 * ct 1120, ss 32.  keygen = DeriveKeyPairPacked (:131-141; the packed sk is the seed itself), encaps = Encapsulate
 * (:173-182, kem.ErrPubKey through status / CB200_ERR_PUBKEY as in cb200_mlkem_encaps), decaps = Decapsulate
 * (:185-191, which re-derives the key pair from the 32-byte sk). */
int cb200_xwing_keygen(const uint8_t *seeds, uint8_t *pk, size_t n);
int cb200_xwing_encaps(const uint8_t *pk, size_t pk_stride, const uint8_t *eseeds, uint8_t *ct, uint8_t *ss,
                       uint8_t *status, size_t n);
int cb200_xwing_decaps(const uint8_t *sk, size_t sk_stride, const uint8_t *ct, uint8_t *ss, size_t n);

/* kem/hybrid (hybrid.go:197-283 over xkem.go): keys, ciphertexts and the 64-byte shared secret are the two halves
 * side by side in the order of hybrid.go:34-62; key seed 64, encapsulation seed 32.
 * status bit 0 = kem.ErrPubKey (non-canonical ML-KEM ek or small-order X25519 share), bit 1 = kem.ErrPrivKey. */
#define CB200_HYBRID_X25519MLKEM768 0  /* ML-KEM-768 || X25519:  pk 1216, sk 2432, ct 1120 */
#define CB200_HYBRID_KYBER768_X25519 1 /* X25519 || Kyber768:    pk 1216, sk 2432, ct 1120 */
#define CB200_HYBRID_KYBER512_X25519 2 /* X25519 || Kyber512:    pk 832,  sk 1664, ct 800  */
int cb200_hybrid_keygen(int id, const uint8_t *seeds, uint8_t *pk, uint8_t *sk, size_t n);
int cb200_hybrid_encaps(int id, const uint8_t *pk, size_t pk_stride, const uint8_t *seeds, uint8_t *ct, uint8_t *ss,
                        uint8_t *status, size_t n);
int cb200_hybrid_decaps(int id, const uint8_t *sk, size_t sk_stride, const uint8_t *ct, uint8_t *ss, uint8_t *status,
                        size_t n);
size_t cb200_hybrid_public_key_size(int id);
size_t cb200_hybrid_private_key_size(int id);
size_t cb200_hybrid_ciphertext_size(int id);

/* ---- ML-DSA (mode = 44, 65 or 87) and round-3 Dilithium (mode = 2, 3 or 5); sign/dilithium/gen.go:80-162 ----
 * Same contracts as the ML-DSA-65 entry points documented below, with the parameter set as first argument:
 *   ML-DSA-44 / 65 / 87 (sign/mldsa/mldsa{44,65,87}):    sk 2560 / 4032 / 4896, pk 1312 / 1952 / 2592, sig 2420 / 3309 / 4627
 *   Dilithium2 / 3 / 5  (sign/dilithium/mode{2,3,5}):     sk 2528 / 4000 / 4864, pk 1312 / 1952 / 2592, sig 2420 / 3293 / 4595
 * Round 3 (NIST = false, internal/params.go:15-17) has no context string (a non-empty one is CB200_ERR_ARG, the
 * reference's sign.ErrContextNotSupported), ignores rnd and flags, and signs the message as given. */
int cb200_mldsa_sign(int mode, const uint8_t *sk, size_t sk_stride, const uint8_t *msgs, const uint64_t *msg_off,
                     const uint8_t *context, size_t ctxlen, const uint8_t *rnd, uint8_t *sig, uint8_t *status, size_t n,
                     int flags, uint64_t *attempts);
int cb200_mldsa_verify(int mode, const uint8_t *pk, size_t pk_stride, const uint8_t *msgs, const uint64_t *msg_off,
                       const uint8_t *context, size_t ctxlen, const uint8_t *sig, uint8_t *ok, size_t n, int flags);
int cb200_mldsa_keygen(int mode, const uint8_t *seeds, uint8_t *pk, uint8_t *sk, size_t n);
size_t cb200_mldsa_public_key_size(int mode);
size_t cb200_mldsa_private_key_size(int mode);
size_t cb200_mldsa_signature_size(int mode);

/* ---- ML-DSA-65 ---- */
/* sign.Scheme.Sign / SignTo    sign/mldsa/mldsa65/dilithium.go:282-303,56-84  ->
 * internal.SignTo (ML-DSA.Sign_internal)  sign/mldsa/mldsa65/internal/dilithium.go:340-470,
 * including (*PrivateKey).Unpack (:142-163): A = ExpandA(rho), NTT(s1), NTT(s2), NTT(t0) are rebuilt on
 * the device (once if sk_stride = 0, else per operation).
 * sk: packed private key(s), 4032 bytes; op i uses sk + i*sk_stride (0 = one key for all).
 * msgs: all messages back to back; message i = msgs[msg_off[i] .. msg_off[i+1]) (n+1 offsets).
 * context/ctxlen: the FIPS 204 context string, shared by the batch (ctxlen <= 255; host pointer).
 * rnd: n x 32 bytes of signing randomness, or NULL for deterministic signing (rnd = 0^32).
 * sig: n x 3309 bytes.  status (optional): n bytes, 1 = the 576-attempt cap was hit (the reference
 * panics there); attempts (optional, host pointer): total rejection-loop iterations of the batch.
 * flags: CB200_SIGN_INTERNAL = ML-DSA.Sign_internal on the message as given (no 0x00||len||ctx framing,
 * the ACVP interface, sign/mldsa/mldsa65/dilithium.go:87-98). */
int cb200_mldsa65_sign(const uint8_t *sk, size_t sk_stride, const uint8_t *msgs, const uint64_t *msg_off,
                       const uint8_t *context, size_t ctxlen, const uint8_t *rnd, uint8_t *sig, uint8_t *status,
                       size_t n, int flags, uint64_t *attempts);
/* sign.Scheme.Verify       sign/mldsa/mldsa65/dilithium.go:305-330,115-138 -> internal.Verify internal/dilithium.go:273-332,
 * including (*PublicKey).Unpack (:113-126): A = ExpandA(rho), tr = H(pk) rebuilt on the device.
 * pk: packed public key(s), 1952 bytes, op i uses pk + i*pk_stride (0 = shared); sig: n x 3309 bytes;
 * ok: n bytes, 1 = valid.  A signature of the wrong length is the caller's (shim's) `false`. */
int cb200_mldsa65_verify(const uint8_t *pk, size_t pk_stride, const uint8_t *msgs, const uint64_t *msg_off,
                         const uint8_t *context, size_t ctxlen, const uint8_t *sig, uint8_t *ok, size_t n, int flags);
/* sign.Scheme.DeriveKey    sign/mldsa/mldsa65/dilithium.go:266-276 -> internal.NewKeyFromSeed internal/dilithium.go:181-241.
 * seeds: n x 32; pk: n x 1952; sk: n x 4032 (packed, = MarshalBinary). */
int cb200_mldsa65_keygen(const uint8_t *seeds, uint8_t *pk, uint8_t *sk, size_t n);
size_t cb200_mldsa65_public_key_size(void);
size_t cb200_mldsa65_signature_size(void);
size_t cb200_mldsa65_private_key_size(void);

#ifdef __cplusplus
}
#endif
#endif
