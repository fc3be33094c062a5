/* curdle_b200 — C ABI of the B200-native BLS12-381 G1 hot path underneath
 * jsign/go-curdleproofs.
 *
 * The reference has no FFI/plugin interface: its hot path is the set of
 * gnark-crypto v0.11.0 methods it calls (SURVEY.md §8b).  Each entry point
 * below names the reference call sites (file:line under /root/reference) whose
 * gnark call it replaces; INTEGRATION.md shows the cgo stubs that bind them.
 *
 * Conventions
 *  - plain C, `extern "C"`, pointers + sizes only; no torch / CUDA types.
 *  - memory layouts are gnark-crypto's, so Go slices cross without copies on
 *    the Go side (`unsafe.Pointer(&s[0])`):
 *      fp.Element  = 6 x uint64 little-endian limbs, Montgomery (R = 2^384)   48 B
 *      fr.Element  = 4 x uint64 little-endian limbs, Montgomery (R = 2^256)   32 B
 *      G1Affine    = {X, Y}      96 B, point at infinity == (0, 0)
 *      G1Jac       = {X, Y, Z}  144 B, point at infinity == Z = 0
 *  - every function returns CDL_OK (0) or a negative cdl_status;
 *    cdl_last_error(ctx) gives a human-readable message for the calling thread's
 *    last failure on that context.
 *  - host-pointer entry points copy in/out and retain nothing after return (cgo
 *    pointer rule).  A context is bound to one CUDA device, or to a list of them
 *    (cdl_create_devices), and is safe to call from many OS threads (calls
 *    serialise on an internal mutex; use one context per thread or the *_batch
 *    entry points for concurrency).
 *  - there is NO CPU fallback: without a CUDA device cdl_create fails with
 *    CDL_ERR_NO_DEVICE.
 */
#ifndef CURDLE_B200_H
#define CURDLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cdl_ctx cdl_ctx;

typedef enum cdl_status {
  CDL_OK = 0,
  CDL_ERR_NO_DEVICE = -1,   /* no CUDA device / driver: the library never falls back to the CPU */
  CDL_ERR_CUDA = -2,        /* a CUDA runtime call failed (see cdl_last_error) */
  CDL_ERR_INVALID_ARG = -3, /* null pointer, bad size, length mismatch (gnark MultiExp's only error) */
  CDL_ERR_DECODE = -4,      /* malformed point / scalar encoding (gnark SetBytes / Decoder error) */
  CDL_ERR_PROTOCOL = -5,    /* reference returns (.., err): zero challenge, bad lengths, "randomizer is zero" */
  CDL_ERR_TOO_LARGE = -6,   /* exceeds a documented size limit of this build */
  CDL_ERR_INTERNAL = -7
} cdl_status;

typedef struct cdl_fp { uint64_t l[6]; } cdl_fp;        /* gnark fp.Element */
typedef struct cdl_fr { uint64_t l[4]; } cdl_fr;        /* gnark fr.Element */
typedef struct cdl_g1_affine { cdl_fp x, y; } cdl_g1_affine;    /* gnark bls12381.G1Affine */
typedef struct cdl_g1_jac { cdl_fp x, y, z; } cdl_g1_jac;       /* gnark bls12381.G1Jac */

/* ---- context ---------------------------------------------------------- */
int32_t cdl_create(int device, cdl_ctx** out);
/* A context whose batched calls use the GPUs devices[0 .. n).  cdl_create(d) is cdl_create_devices(&d, 1).
 * Each entry is a device slot with its own lanes (cdl_set_lanes = lanes per slot), pools and CRS replicas;
 * a device may be listed more than once.  Results never depend on the device list.
 *
 * Split over the slots: the batched Whisk shuffle-proof calls, cdl_shuffle_permute_commit_batch,
 * cdl_prove_batch, cdl_verify_batch, the batched tracker-proof calls and cdl_whisk_match_trackers.  Slot s
 * of the D' = max(1, min(n, B / 32)) slots in use takes the contiguous block s of B instances (block sizes
 * differ by at most one, as sharding.shard_bounds deals them; for matching the block bounds are rounded to
 * multiples of 256 trackers and every slot matches its block against all keys), and cuts it into lanes
 * as a one-device context cuts a batch.  A call of fewer than 64 instances, and every single
 * (non-batched) protocol call, runs on slot 0.
 *
 * Single calls split by size, each slot running its block on its lane 0 (one piece per slot):
 * cdl_g1_msm of more than 1 024 terms (and cdl_g1_sum_affine through it) over D' = max(1, min(n, terms /
 * 65 536)) slots, so from 131 072 terms on; slot s sums its contiguous block of the terms and the D' partial
 * sums are added on devices[0].  cdl_g1_batch_scalar_mul_base over D' = max(1, min(n, scalars / 32 768))
 * slots, so from 65 536 scalars on; slot s multiplies its contiguous block with its own cached tables.
 * cdl_whisk_generate_registration_batch likewise over D' = max(1, min(n, B / 6 554)) slots, in blocks of
 * validators.  The elementwise calls split by points the same way, each with its own minimum block kMin
 * over D' = max(1, min(n, points / kMin)) slots: cdl_g1_decompress (16 384), cdl_g1_compress (131 072),
 * cdl_g1_batch_to_affine (32 768), cdl_g1_scalar_mul_affine (4 096) and cdl_g1_fold (4 096); slot s writes
 * its contiguous range of the outputs.  cdl_g1_msm_batch splits at MSM boundaries over D' = max(1, min(n,
 * terms / 65 536)) slots: slot s takes whole, contiguous MSMs, the blocks balanced by terms, and a call whose
 * terms all sit in one MSM does not split.  Below 2 * kMin units every one of these calls runs on slot 0
 * exactly as on a one-device context.  A split call returns what the one-device call returns: the same
 * bytes, status, return code and cdl_last_error text.  Its blocks read their inputs and write their outputs
 * concurrently, so outputs may be the inputs themselves (in place) but must not overlap them otherwise.
 *
 * Everything else runs on slot 0's device (devices[0]): cdl_g1_msm and cdl_g1_sum_affine of at most 1 024
 * terms, the entry points on device vectors (*_device, including cdl_g1_msm_batch_device), the sharded MSMs,
 * cdl_dev_* buffers (device memory of devices[0]), cdl_fp_mul, cdl_rand_get_g1_affines and CRS generation.
 * cdl_comm_init refuses a context of more than one slot: the NCCL-sharded MSM runs one process (and
 * one single-device context) per GPU.
 * CDL_ERR_INVALID_ARG for n == 0, n > 16 or a device id out of range; CDL_ERR_NO_DEVICE without a
 * CUDA device. */
int32_t cdl_create_devices(const int32_t* devices, size_t n, cdl_ctx** out);
/* The device list of the context: *n receives its length, devices[0 .. min(cap, *n)) its entries. */
int32_t cdl_context_devices(cdl_ctx* ctx, int32_t* devices, size_t cap, size_t* n);
void cdl_destroy(cdl_ctx* ctx);
const char* cdl_last_error(cdl_ctx* ctx);
/* ABI version of this build (major << 16 | minor). */
uint32_t cdl_abi_version(void);
/* Device description: SM count and name (diagnostics / bench). */
int32_t cdl_device_info(cdl_ctx* ctx, int32_t* sm_count, int32_t* clock_khz, char* name, size_t name_cap);

/* ---- 1:1 gnark replacements, host pointers ----------------------------- */

/* (*G1Jac).MultiExp(points, scalars, cfg): out = sum scalars[i] * points[i].
 * Replaces all 39 call sites, e.g. curdleproof.go:72,75,109,113;
 * msmaccumulator/msmaccumulator.go:59; innerproductargument.go:65,69,108,121,125,138;
 * samemultiscalarargument.go:63-72,93-111; common/util.go:75,82.
 * Infinity bases are skipped; n == 0 gives infinity.  The result is returned
 * normalised (Z = 1, or Z = 0 for infinity) — any representative is valid
 * because only canonical encodings are observable (SURVEY.md §8c).
 * CDL_ERR_TOO_LARGE for n >= 2^30 (on a context of several device slots before any input is read).  Above
 * 1 024 terms the per-device limits - the batch-affine scratch budget (the MSM falls back to extended-Jacobian
 * buckets beyond it), 2^32 sorted bucket entries (CDL_ERR_TOO_LARGE) and device allocation (CDL_ERR_CUDA) -
 * apply to the whole MSM on a one-device context and to each slot's block on a split call
 * (cdl_create_devices), so a split call fails nowhere a one-device call succeeds and may succeed where one
 * device alone reaches a limit.  The 144 output bytes are the same either way. */
int32_t cdl_g1_msm(cdl_ctx* ctx, const cdl_g1_affine* points, const cdl_fr* scalars, size_t n, cdl_g1_jac* out);

/* k independent MSMs in one launch; MSM j covers points/scalars
 * [offsets[j], offsets[j+1]).  Affine results.  Covers the 4 / 6 MSMs of one
 * IPA / SameMSM round (innerproductargument.go:108-138,
 * samemultiscalarargument.go:93-111) and the verifier's tiny MSMs
 * (innerproductargument.go:238,250,275,281).
 * CDL_ERR_INVALID_ARG for offsets that decrease or when k + offsets[k] >= 2^30 (the point pool), before any
 * input is read.  On a context of several device slots, from 2 * 65 536 terms held by at least two MSMs, the
 * MSMs are dealt to the slots in contiguous groups of whole MSMs balanced by terms (cdl_create_devices). */
int32_t cdl_g1_msm_batch(cdl_ctx* ctx, const cdl_g1_affine* points, const cdl_fr* scalars,
                         const uint32_t* offsets, size_t k, cdl_g1_affine* out);

/* (*G1Affine).ScalarMultiplication for n points: out[i] = s[i*scalar_stride] * in[i].
 * scalar_stride == 0 broadcasts one scalar: the Whisk rescale Ts[i] = k*Rs[i]
 * (common/util.go:55-63); scalar_stride == 1 gives per-element scalars:
 * Gs'[i] = beta^-(i+1) * Gs[i] (grandproductargument.go:94-103).  The scalar is
 * the fr.Element itself (the reference converts it with common.FrToBigInt,
 * common/util.go:16-20).  Split by points from 2 * 4 096 points on a context of several device slots; a
 * broadcast scalar goes to every block. */
int32_t cdl_g1_scalar_mul_affine(cdl_ctx* ctx, const cdl_g1_affine* in, const cdl_fr* s, size_t n,
                                 size_t scalar_stride, cdl_g1_affine* out);

/* Base folding L[i] += x * R[i], i < n, result affine in place.
 * Replaces the serial loops innerproductargument.go:155-166 (called with x =
 * gamma for G and gamma^-1 for G') and samemultiscalarargument.go:129-135.
 * Split by points from 2 * 4 096 points on a context of several device slots. */
int32_t cdl_g1_fold(cdl_ctx* ctx, cdl_g1_affine* L, const cdl_g1_affine* R, const cdl_fr* x, size_t n);

/* bls12381.BatchScalarMultiplicationG1: out[i] = scalars[i] * base, i < n, for one base and many scalars: the
 * k-commitments kG and initial trackers (G, kG) of many validators, or the blinder products r * G of tracker
 * proofs.  Scalars are gnark fr.Elements (Montgomery), read as cdl_g1_scalar_mul_affine reads them (limbs
 * >= r included).  out receives affine points in gnark's layout (infinity = (0, 0)) and out48 the 48-byte
 * compressed encodings cdl_g1_compress gives; either may be NULL, not both.  For every input the output
 * bytes equal those of cdl_g1_scalar_mul_affine on n copies of base with scalar_stride = 1.
 * base must be on the curve and in G1 (checked on the device with decompression's subgroup test), else
 * CDL_ERR_INVALID_ARG with a message; the point at infinity gives infinity for every scalar.
 * Two device paths, chosen by n and the context's table cache, with the same results: from
 * the base's width-12 fixed-base table (22 x 2 048 points, 4.3 MB; 22 mixed additions per scalar), used
 * when that table is cached or n is large enough that building it pays off (the table is then built and
 * cached); otherwise GLV scalar multiplication of every scalar, which builds no table.  The context keeps
 * the tables of its 4 most recently used bases per device slot (about 17 MB of device memory per slot,
 * freed by cdl_destroy); a base whose table is cached is not checked again.  Scalars travel in chunks of 2^20.
 * On a context of several slots a call of 65 536 scalars or more is split (cdl_create_devices): every slot
 * in use runs its block with its own cache, checks the base when its table is not cached and picks its path
 * by its block size and its cache alone; a smaller call runs on the context's own cache.  Device 0 can
 * therefore hold both caches (up to 8 tables).  A rejected base fails every block alike, before any output
 * is written.
 * n == 0 does nothing; CDL_ERR_INVALID_ARG for a null ctx, base or scalars or when both outputs are NULL;
 * CDL_ERR_TOO_LARGE when n exceeds CDL_BASE_MUL_MAX, before any input is read. */
#define CDL_BASE_MUL_MAX (1u << 24)
int32_t cdl_g1_batch_scalar_mul_base(cdl_ctx* ctx, const cdl_g1_affine* base, const cdl_fr* scalars, size_t n,
                                     cdl_g1_affine* out, uint8_t* out48);

/* bls12381.BatchJacobianToAffineG1 (transcript/transcript.go:26 and every Serialize).  Split by points from
 * 2 * 32 768 points on a context of several device slots. */
int32_t cdl_g1_batch_to_affine(cdl_ctx* ctx, const cdl_g1_jac* in, size_t n, cdl_g1_affine* out);

/* sum of n affine points (crs.go:41-48 Gsum / Hsum). */
int32_t cdl_g1_sum_affine(cdl_ctx* ctx, const cdl_g1_affine* in, size_t n, cdl_g1_affine* out);

/* G1Affine.Bytes() for n points -> n * 48 compressed bytes
 * (transcript/transcript.go:35, whisk/types.go:79-84).  Split by points from 2 * 131 072 points on a
 * context of several device slots. */
int32_t cdl_g1_compress(cdl_ctx* ctx, const cdl_g1_affine* in, size_t n, uint8_t* out48);

/* G1Affine.SetBytes on n 48-byte compressed encodings, with curve and
 * subgroup checks (whisk/types.go:86-95; Decoder in curdleproof.go:320-356).
 * status[i] == 0 on success, else a positive reason code (1 bad flags /
 * uncompressed, 2 non-canonical x, 3 no square root, 4 not in subgroup,
 * 5 bad infinity padding).  Returns CDL_ERR_DECODE if any point failed; cdl_last_error then names the
 * first rejected point.  Every point and status is written either way.  Split by points from 2 * 16 384
 * points on a context of several device slots, with the same statuses, return code and message. */
int32_t cdl_g1_decompress(cdl_ctx* ctx, const uint8_t* in48, size_t n, cdl_g1_affine* out, uint8_t* status);

/* ---- protocol level: the reference's public API, batched on the GPU ------
 * The Go types with unexported fields (curdleproof.Proof, whisk.*Bytes) cross
 * this boundary in their own wire format (curdleproof.go:358-387,
 * whisk/types.go:53-72); INTEGRATION.md shows the Go-side wrappers.  Group
 * elements never touch the host except as 48-byte encodings; the host side of
 * these calls is the Merlin transcript, Fiat-Shamir challenges, Fr arithmetic
 * and the RNG, exactly the split north_star describes.                        */

typedef struct cdl_rand cdl_rand; /* common.Rand (common/rand.go:13-33) */
typedef struct cdl_crs cdl_crs;   /* curdleproof.CRS (crs.go:10-18), device resident */

#define CDL_N_BLINDERS 4                    /* common/constants.go:3 */
#define CDL_WHISK_SHUFFLE_PROOF_SIZE 4576   /* whisk/types.go:21 */
#define CDL_WHISK_TRACKER_SIZE 96           /* WhiskTracker{rG, krG}: 2 x 48 B, whisk/types.go:74-77 */

/* common.NewRand / GetFr(s) / GetG1Affines / GeneratePermutation (common/rand.go:19-113) */
int32_t cdl_rand_new(uint64_t seed, cdl_rand** out);
void cdl_rand_free(cdl_rand* r);
int32_t cdl_rand_get_frs(cdl_rand* r, size_t n, cdl_fr* out);
int32_t cdl_rand_get_g1_affines(cdl_ctx* ctx, cdl_rand* r, size_t n, cdl_g1_affine* out);
int32_t cdl_rand_generate_permutation(cdl_rand* r, size_t n, uint32_t* out);

/* curdleproof.GenerateCRS (crs.go:20-59): draws ell Gs, 4 Hs, H, Gt, Gu and forms Gsum, Hsum. */
int32_t cdl_crs_generate(cdl_ctx* ctx, size_t ell, cdl_rand* r, cdl_crs** out);
/* Wrap an existing Go-side CRS: points[] = Gs[ell] | Hs[4] | H | Gt | Gu | Gsum | Hsum, all affine.
 * Gsum must be the sum of the Gs and Hsum the sum of the Hs (one MSM of ell + 4 terms checks both):
 * the prover and verifier use the sums in place of the vectors, so a CRS whose sums disagree would give
 * proofs that differ from the reference's and that its verifier rejects.  CDL_ERR_INVALID_ARG otherwise,
 * with cdl_last_error naming the wrong sum.  The points are not checked to be on the curve or in G1. */
int32_t cdl_crs_from_points(cdl_ctx* ctx, size_t ell, const cdl_g1_affine* points, cdl_crs** out);
/* Same order as cdl_crs_from_points, ell + 9 points. */
int32_t cdl_crs_export(cdl_ctx* ctx, const cdl_crs* crs, cdl_g1_affine* points);
size_t cdl_crs_ell(const cdl_crs* crs);
/* Fixed-base tables for the CRS points: protocol calls of at least `instances` proofs (per lane of a
 * batched call) sum their multiples of Gs, Hs, H, Gt, Gu, Gsum, Hsum from tables of d * 2^(12 w) * P
 * (4.3 MB per point, built on the device the first time a CRS is used that way and owned by the CRS
 * object) instead of running buckets / double-and-add over them.  -1 = default (environment
 * CDL_FIXED_BASE_MINB, else 64), 0 = never.  Tuning aid; results do not depend on it. */
int32_t cdl_set_fixed_base_min_batch(cdl_ctx* ctx, int32_t instances);
/* Batched Whisk shuffle-proof verification (cdl_whisk_is_valid_shuffle_proof_batch): a lane of at least
 * `proofs` proofs first checks all of its proofs' final verifier equations at once, as one large MSM over a
 * random linear combination of them (128-bit weights derived from the batch; a false pass has probability
 * at most 2^-128).  When that sum is not the point at infinity, the proofs are checked one by one as
 * without it.  -1 = default (64), 0 = never.  Tuning aid; results do not depend on it. */
int32_t cdl_set_batch_verify_min(cdl_ctx* ctx, int32_t proofs);
void cdl_crs_free(cdl_crs* crs);

/* common.ShufflePermuteCommit (common/util.go:45-88): Ts = perm(k*Rs), Us = perm(k*Ss),
 * M = <perm(0..ell-1), Gs> + <rs_m, Hs> with rs_m = 4 fresh Fr from r. */
int32_t cdl_shuffle_permute_commit(cdl_ctx* ctx, const cdl_crs* crs, const cdl_g1_affine* Rs, const cdl_g1_affine* Ss,
                                   const uint32_t* perm, const cdl_fr* k, cdl_rand* r, cdl_g1_affine* Ts,
                                   cdl_g1_affine* Us, cdl_g1_jac* M, cdl_fr* rs_m);

/* curdleproof.Prove (curdleproof.go:38-197) followed by Proof.Serialize (:358-387).
 * proof_len receives the serialized size (18 + 10m points, 7 scalars, 10 length prefixes). */
int32_t cdl_prove(cdl_ctx* ctx, const cdl_crs* crs, const cdl_g1_affine* Rs, const cdl_g1_affine* Ss,
                  const cdl_g1_affine* Ts, const cdl_g1_affine* Us, const cdl_g1_jac* M, const uint32_t* perm,
                  const cdl_fr* k, const cdl_fr* rs_m, cdl_rand* r, uint8_t* proof, size_t proof_cap,
                  size_t* proof_len);

/* Proof.FromReader (curdleproof.go:320-356) + curdleproof.Verify (:199-318).
 * *ok = 1 / 0 is the reference's bool; a non-zero return is the reference's error
 * (CDL_ERR_DECODE for malformed bytes, CDL_ERR_PROTOCOL e.g. "randomizer is zero"). */
int32_t cdl_verify(cdl_ctx* ctx, const cdl_crs* crs, const uint8_t* proof, size_t proof_len,
                   const cdl_g1_affine* Rs, const cdl_g1_affine* Ss, const cdl_g1_affine* Ts,
                   const cdl_g1_affine* Us, const cdl_g1_jac* M, cdl_rand* r, int32_t* ok);

/* Batched forms of the three calls above: B caller-supplied instances in lock step, one GPU launch per
 * protocol stage for the whole batch, cut into lanes (cdl_set_lanes) as the Whisk batch calls are.
 * Arrays are instance-major: Rs, Ss, Ts, Us and perms hold B x ell entries; ks, M, rands, status, ok and
 * proof_lens B entries; rs_m B x 4.  Proof b is at proofs + b * proof_cap (proof_stride for verification,
 * where proof_lens[b] <= proof_stride).  For every instance b the batch gives what the single call gives on
 * the same inputs: the same outputs, status[b] equal to the single call's return code and the same position
 * of rands[b] afterwards.  An instance whose status is not CDL_OK leaves its outputs as they were, except
 * proof_lens[b] when the proof did not fit proof_cap; an instance with a permutation entry >= ell or a
 * proof that fails to decode draws nothing from its Rand.  Returns CDL_OK when the arguments are valid,
 * whatever the per-instance statuses (cdl_last_error then holds a failing instance's message);
 * CDL_ERR_INVALID_ARG for a null pointer, B == 0 or a CRS of another context; CDL_ERR_TOO_LARGE when one
 * lane's instances would need 2^30 or more pool points (about 150 000 instances at ell = 508). */
int32_t cdl_shuffle_permute_commit_batch(cdl_ctx* ctx, const cdl_crs* crs, size_t B, const cdl_g1_affine* Rs,
                                         const cdl_g1_affine* Ss, const uint32_t* perms, const cdl_fr* ks,
                                         cdl_rand* const* rands, cdl_g1_affine* Ts, cdl_g1_affine* Us, cdl_g1_jac* M,
                                         cdl_fr* rs_m, int32_t* status);
int32_t cdl_prove_batch(cdl_ctx* ctx, const cdl_crs* crs, size_t B, const cdl_g1_affine* Rs, const cdl_g1_affine* Ss,
                        const cdl_g1_affine* Ts, const cdl_g1_affine* Us, const cdl_g1_jac* M, const uint32_t* perms,
                        const cdl_fr* ks, const cdl_fr* rs_m, cdl_rand* const* rands, uint8_t* proofs,
                        size_t proof_cap, size_t* proof_lens, int32_t* status);
int32_t cdl_verify_batch(cdl_ctx* ctx, const cdl_crs* crs, size_t B, const uint8_t* proofs, size_t proof_stride,
                         const size_t* proof_lens, const cdl_g1_affine* Rs, const cdl_g1_affine* Ss,
                         const cdl_g1_affine* Ts, const cdl_g1_affine* Us, const cdl_g1_jac* M,
                         cdl_rand* const* rands, int32_t* ok, int32_t* status);

/* whisk.GenerateWhiskShuffleProof (whisk/whisk.go:63-114).  Trackers are
 * 96-byte {rG, krG} pairs; crs ell trackers in, ell out; proof is zero padded
 * to proof_cap (4576 for the reference's N = 128). */
int32_t cdl_whisk_generate_shuffle_proof(cdl_ctx* ctx, const cdl_crs* crs, const uint8_t* pre_trackers,
                                         cdl_rand* r, uint8_t* post_trackers, uint8_t* proof, size_t proof_cap);
/* whisk.IsValidWhiskShuffleProof (whisk/whisk.go:20-61). */
int32_t cdl_whisk_is_valid_shuffle_proof(cdl_ctx* ctx, const cdl_crs* crs, const uint8_t* pre_trackers,
                                         const uint8_t* post_trackers, size_t n_pre, size_t n_post,
                                         const uint8_t* proof, size_t proof_len, cdl_rand* r, int32_t* ok);

/* Batched forms: B independent instances advance in lock step, one GPU launch
 * per protocol stage for the whole batch (config 4 of BASELINE.json).  Arrays
 * are instance-major; status[b] is the per-instance return code. */
int32_t cdl_whisk_generate_shuffle_proof_batch(cdl_ctx* ctx, const cdl_crs* crs, size_t B,
                                               const uint8_t* pre_trackers, cdl_rand* const* rands,
                                               uint8_t* post_trackers, uint8_t* proofs, size_t proof_cap,
                                               int32_t* status);
int32_t cdl_whisk_is_valid_shuffle_proof_batch(cdl_ctx* ctx, const cdl_crs* crs, size_t B,
                                               const uint8_t* pre_trackers, const uint8_t* post_trackers,
                                               const uint8_t* proofs, size_t proof_len, cdl_rand* const* rands,
                                               int32_t* ok, int32_t* status);
/* whisk.GenerateWhiskTrackerProof (whisk/whisk.go:149-176), batched over B validators: tracker b is
 * 96 bytes {rG, krG}, ks[b] the secret, one blinder is drawn from rands[b]; proofs receives B x 128
 * bytes (A | B | s, whisk/types.go:98-127).  status[b] = CDL_ERR_DECODE when the tracker does not decode. */
#define CDL_WHISK_TRACKER_PROOF_SIZE 128
int32_t cdl_whisk_generate_tracker_proof_batch(cdl_ctx* ctx, size_t B, const uint8_t* trackers, const cdl_fr* ks,
                                               cdl_rand* const* rands, uint8_t* proofs, int32_t* status);
/* whisk.IsValidWhiskTrackerProof (whisk/whisk.go:116-147): k_comms holds B x 48 bytes (kG).
 * ok[b] is the reference's bool, status[b] its error (CDL_ERR_DECODE for malformed proof / points). */
int32_t cdl_whisk_is_valid_tracker_proof_batch(cdl_ctx* ctx, size_t B, const uint8_t* trackers, const uint8_t* k_comms,
                                               const uint8_t* proofs, int32_t* ok, int32_t* status);
/* Whisk registration material for B validators (first-proposal registration, checked by
 * process_whisk_registration): for validator b with secret ks[b] (gnark fr.Element, read as
 * cdl_whisk_generate_tracker_proof_batch reads it, limbs >= r included), r = the next Fr drawn from rands[b];
 * trackers + 96 b = {r*G, k*r*G} compressed, k_comms + 48 b = k*G, proofs + 128 b = the opening proof that
 * cdl_whisk_generate_tracker_proof_batch gives for that tracker and k with rands[b] as left after drawing r
 * (it draws one blinder).  The bytes and the Rand positions are those of that composition (draw r,
 * cdl_g1_batch_scalar_mul_base, cdl_g1_scalar_mul_affine, cdl_g1_batch_scalar_mul_base for k*G, then the proof
 * call), but every point is a multiple of G (k*r and blinder*r are formed on the host), so the call is one
 * fixed-base multiplication of 5 B scalars by G, from G's cached table as cdl_g1_batch_scalar_mul_base runs it.
 * rands[b] must be a distinct Rand per validator (the validators draw concurrently; a Rand listed twice races).
 * status[b] = CDL_ERR_PROTOCOL when r is 0 or 1 (rG at infinity or rG == G); such a validator draws no blinder
 * and its outputs are left as they were.
 * On a context of several device slots a call of at least 2 * 6 554 validators is split (cdl_create_devices),
 * each slot multiplying the 5 * 6 554 or more scalars of its block; the results do not depend on the device list.
 * Returns CDL_OK when the arguments are valid, whatever the statuses; CDL_ERR_INVALID_ARG for a null pointer
 * or B == 0; CDL_ERR_TOO_LARGE for B > CDL_WHISK_REGISTER_MAX, before any Rand is drawn. */
#define CDL_WHISK_REGISTER_MAX (1u << 21)
int32_t cdl_whisk_generate_registration_batch(cdl_ctx* ctx, size_t B, const cdl_fr* ks, cdl_rand* const* rands,
                                              uint8_t* trackers, uint8_t* k_comms, uint8_t* proofs,
                                              int32_t* status);
/* Which of the caller's Whisk secrets own which trackers.  trackers: T x 96 bytes {rG, krG} as in
 * cdl_whisk_generate_tracker_proof_batch; ks: V secrets (gnark fr.Element, Montgomery).
 * owner[t] = the smallest v with ks[v] * rG_t == krG_t (equal as group elements), else -1.
 * status[t] = CDL_OK, CDL_ERR_DECODE when either point fails SetBytes (flags, curve, subgroup),
 * or CDL_ERR_PROTOCOL when rG_t is the point at infinity (such a tracker identifies nobody).
 * owner[t] = -1 whenever status[t] != CDL_OK.  Returns CDL_OK when the arguments are valid,
 * whatever the per-tracker statuses; CDL_ERR_INVALID_ARG for a null pointer, T == 0 or V == 0;
 * CDL_ERR_TOO_LARGE when T or V exceeds CDL_WHISK_MATCH_MAX (2^24).  The reference leaves this
 * check (k * rG == krG, one ScalarMultiplication per pair) to its caller. */
#define CDL_WHISK_MATCH_MAX (1u << 24)
int32_t cdl_whisk_match_trackers(cdl_ctx* ctx, size_t T, const uint8_t* trackers,
                                 size_t V, const cdl_fr* ks, int32_t* owner, int32_t* status);

/* Host-side self test (no GPU needed): out32 receives Merlin's published
 * "test protocol" challenge computed by the library's transcript code;
 * fr_out receives (a*b + a - b)^-1 * a^5 computed by the host Fr code. */
int32_t cdl_host_selftest(uint8_t* out32, const cdl_fr* a, const cdl_fr* b, cdl_fr* fr_out);
/* Host-side self test of the eight-way transcript hashing (no GPU needed): n Merlin transcripts and
 * SHAKE256 streams (transcript/transcript.go, common/rand.go) with per-index messages and `rounds`
 * rejection-sampled challenges each, run once one at a time and once as cooperating fibers whose
 * Keccak permutations are batched eight at a time (AVX-512); digest32 receives a hash over all the
 * challenges.  Returns CDL_OK when both runs agree byte for byte; *used_x8 tells whether the
 * eight-way path was available on this host (0: both runs were scalar). */
int32_t cdl_host_selftest_fibers(uint32_t n, uint32_t rounds, uint8_t* digest32, int32_t* used_x8);
/* Per kernel class statistics of the protocol-level calls, of the batched MSMs
 * (cdl_g1_msm_batch, cdl_g1_msm_batch_device, cdl_g1_msm up to 1 024 terms), of
 * cdl_whisk_match_trackers and of cdl_g1_batch_scalar_mul_base since the last reset (class 0
 * small-MSM, 1 elementwise scalar-mul/fold, tracker matching and fixed-base scalar
 * multiplication, 2 decompress, 3 compress / normalise): launches, CUDA-event milliseconds on the
 * launching stream, algorithmic modmul (SURVEY.md §8d conventions; 3 193 per matched (key, tracker)
 * pair and per scalar of cdl_g1_batch_scalar_mul_base, which counts one class-1 launch per chunk of
 * up to 2^20 scalars; cdl_whisk_generate_registration_batch counts as that call on its 5 B scalars) and
 * algorithmic bytes.  Each output array has 4 entries. */
int32_t cdl_engine_stats(cdl_ctx* ctx, uint64_t* launches, double* ms, double* modmul, double* bytes, int reset);
/* Device busy time since the last cdl_engine_stats(.., reset = 1): the length of
 * the union of all timed kernel intervals over every lane's stream (lanes overlap,
 * so the per-class sums above can exceed it).  With several device slots, the
 * largest busy time of one slot. */
int32_t cdl_engine_busy_ms(cdl_ctx* ctx, double* busy_ms);
/* Device busy time of slot `slot` since the last stats reset (union of that slot's lanes' kernel intervals).
 * CDL_ERR_INVALID_ARG for a slot beyond the device list. */
int32_t cdl_engine_busy_ms_device(cdl_ctx* ctx, size_t slot, double* busy_ms);
/* A batched protocol call is cut into up to `lanes` sub-batches (default 4, at
 * least 32 instances each) that advance concurrently on their own CUDA streams
 * and host threads: one lane's host-side transcript work overlaps the other
 * lanes' kernels.  Results do not depend on it.  Also environment CDL_LANES.
 * With several device slots this is the number of lanes per slot. */
int32_t cdl_set_lanes(cdl_ctx* ctx, int32_t lanes);
/* Number of GPU kernels launched by protocol-level calls, batched MSMs, tracker matching,
 * cdl_g1_batch_scalar_mul_base and cdl_whisk_generate_registration_batch on this context so far, summed over
 * its device slots. */
uint64_t cdl_launch_count(cdl_ctx* ctx);

/* ---- large MSM, device-resident vectors, multi-GPU ----------------------
 * cdl_g1_msm switches to a signed-digit Pippenger (on-GPU counting sort of
 * bucket indices, thread-per-bucket XYZZ accumulation, chunked bucket
 * reduction) above 1024 terms; the entry points below expose the same kernel
 * chain on device-resident vectors and across the GPUs of one box
 * (BASELINE.json config 5; gnark's MultiExp is what it replaces, e.g.
 * msmaccumulator/msmaccumulator.go:59, common/util.go:75).                  */

/* Raw device buffers on the context's GPU, for vectors that stay in HBM between
 * calls (a CRS, the sweep's point vectors).  Plain cudaMalloc'ed memory: a host
 * that already owns device memory (another CUDA library, a torch tensor) passes
 * its own pointers to the *_device entry points instead. */
int32_t cdl_dev_alloc(cdl_ctx* ctx, size_t bytes, void** d_ptr);
int32_t cdl_dev_free(cdl_ctx* ctx, void* d_ptr);
int32_t cdl_dev_upload(cdl_ctx* ctx, void* d_dst, const void* h_src, size_t bytes);
int32_t cdl_dev_download(cdl_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);

/* (*G1Affine).ScalarMultiplication on device vectors (common/util.go:55-63), in place allowed. */
int32_t cdl_g1_scalar_mul_affine_device(cdl_ctx* ctx, const cdl_g1_affine* d_in, const cdl_fr* d_s, size_t n,
                                        size_t scalar_stride, cdl_g1_affine* d_out);

/* Base folding L[i] += x * R[i] on device vectors (innerproductargument.go:155-166,
 * samemultiscalarargument.go:129-135); d_x points to one fr.Element in device memory. */
int32_t cdl_g1_fold_device(cdl_ctx* ctx, cdl_g1_affine* d_L, const cdl_g1_affine* d_R, const cdl_fr* d_x, size_t n);

/* (*G1Jac).MultiExp for k independent MSMs whose BASES STAY ON THE DEVICE: term t of MSM j is
 * scalars[t] * d_pool[idx[t]] (bit 31 of idx[t] negates the base; pool indices are below 2^30), t in [offsets[j], offsets[j+1]).
 * idx / scalars / offsets / out_slot are HOST arrays - what the Go orchestration computes between
 * rounds - while d_pool is a device array of affine points (cdl_dev_alloc + cdl_dev_upload, folded in
 * place with cdl_g1_fold_device), so the folded base vectors of innerproductargument.go:100-172 and
 * samemultiscalarargument.go:85-140 never cross PCIe.  Result j is written to d_pool[out_slot[j]]
 * (if out_slot != NULL), to out[j] (affine, if out != NULL) and to out48 + 48*j as the compressed
 * encoding transcript.AppendPoints hashes (if out48 != NULL). */
int32_t cdl_g1_msm_batch_device(cdl_ctx* ctx, cdl_g1_affine* d_pool, const uint32_t* idx, const cdl_fr* scalars,
                                const uint32_t* offsets, size_t k, const uint32_t* out_slot, cdl_g1_affine* out,
                                uint8_t* out48);

/* (*G1Jac).MultiExp on device vectors.  part_index / part_count select the
 * windows part_index, part_index + part_count, ... of the signed-digit
 * decomposition (0 / 1 = the whole MSM); the partial sum is returned already
 * shifted, so partial sums of all parts add up to the MSM.  normalize != 0
 * returns (x, y, 1) or (1, 1, 0).  *kernel_ms (optional) receives the CUDA-event
 * time of the kernel chain on the context's stream.  Synchronous. */
int32_t cdl_g1_msm_device(cdl_ctx* ctx, const cdl_g1_affine* d_points, const cdl_fr* d_scalars, size_t n,
                          uint32_t part_index, uint32_t part_count, int32_t normalize, cdl_g1_jac* d_out,
                          float* kernel_ms);
/* Override the Pippenger window width (2..18 bits; 0 = choose by size).  Tuning aid;
 * the result does not depend on it.  Also settable as environment CDL_MSM_C. */
int32_t cdl_set_msm_window(cdl_ctx* ctx, int32_t window_bits);
/* Number of batch-affine rounds of the large MSM's bucket accumulation (0..8; -1 = choose by the
 * mean bucket load; 0 = extended-Jacobian buckets only): for `rounds` rounds neighbouring summands
 * of every bucket are added as affine points whose inversions are shared by Montgomery's trick
 * (what gnark-crypto's MultiExp does for its large windows).  Tuning aid; the result does not
 * depend on it.  Also settable as environment CDL_MSM_BATCH_AFFINE. */
int32_t cdl_set_msm_batch_affine(cdl_ctx* ctx, int32_t rounds);

/* One process per GPU: rank 0 calls cdl_comm_unique_id, the host application
 * ships the 128 bytes to every rank (any transport), every rank calls
 * cdl_comm_init (collective; NCCL over NVLink / NVSwitch, bound with dlopen)
 * on a single-device context (CDL_ERR_INVALID_ARG with more than one slot). */
int32_t cdl_comm_unique_id(uint8_t* id128);
int32_t cdl_comm_init(cdl_ctx* ctx, const uint8_t* id128, int32_t rank, int32_t world);
int32_t cdl_comm_destroy(cdl_ctx* ctx);
/* Which windows rank `rank` of `world` owns for an MSM of n terms (window_bits 0 = choose by size). */
void cdl_comm_partition(size_t n, int32_t world, int32_t rank, int32_t window_bits, int32_t* first_window,
                        int32_t* window_step, int32_t* n_windows, int32_t* my_windows);
/* Window-partitioned MSM: every rank passes the same (replicated) vectors, sums
 * its own windows, the partial sums (one 144-byte point per rank) are
 * all-gathered with NCCL and added on every rank; every rank receives the
 * normalised result.  Collective over the communicator of cdl_comm_init
 * (world == 1 needs no communicator). */
int32_t cdl_g1_msm_sharded_device(cdl_ctx* ctx, const cdl_g1_affine* d_points, const cdl_fr* d_scalars, size_t n,
                                  cdl_g1_jac* d_out, float* kernel_ms);
int32_t cdl_g1_msm_sharded(cdl_ctx* ctx, const cdl_g1_affine* points, const cdl_fr* scalars, size_t n,
                           cdl_g1_jac* out);

/* ---- diagnostics / roofline ------------------------------------------- */
/* out[i] = a[i] * b[i] in Fp (Montgomery).  K1 of SURVEY.md §7. */
int32_t cdl_fp_mul(cdl_ctx* ctx, const cdl_fp* a, const cdl_fp* b, size_t n, cdl_fp* out);
/* Integer-pipe peak microbenchmarks (SURVEY.md §7 step 0).  kind 0: independent
 * 32-bit IMAD chains; 1: mad.wide (IMAD.WIDE) chains; 2: dependent Fp
 * Montgomery products (practical modmul peak).  Writes the measured ops/s
 * (IMAD/s for 0-1, modmul/s for 2) and the kernel time. */
int32_t cdl_int_peak(cdl_ctx* ctx, int kind, int iters, double* ops_per_s, double* ms);
/* Same with an explicit launch shape (blocks per SM, threads per block) and two more
 * kinds: 3 / 4 = two / three independent product chains per thread (ILP probes). */
int32_t cdl_int_peak_cfg(cdl_ctx* ctx, int kind, int iters, int blocks_per_sm, int threads_per_block,
                         double* ops_per_s, double* ms);

#ifdef __cplusplus
}
#endif
#endif /* CURDLE_B200_H */
