package gpu

/*
#include "curdle_b200.h"
*/
import "C"

import (
	"unsafe"

	bls12381 "github.com/consensys/gnark-crypto/ecc/bls12-381"
	"github.com/consensys/gnark-crypto/ecc/bls12-381/fr"
)

// Rand is common.Rand (common/rand.go): the same SHAKE256 stream with the same rejection sampling,
// owned by the library so that the draw order a caller observes across CRS generation, proof
// generation and validation (whisk/whisk_test.go:36-50) is the reference's.
type Rand struct{ h *C.cdl_rand }

// NewRand is common.NewRand(seed).
func NewRand(seed uint64) (*Rand, error) {
	var h *C.cdl_rand
	if rc := C.cdl_rand_new(C.uint64_t(seed), &h); rc != 0 {
		return nil, errStatus(rc)
	}
	return &Rand{h}, nil
}

// Free releases the generator.
func (r *Rand) Free() { C.cdl_rand_free(r.h) }

// GetFrs is (*Rand).GetFrs.
func (r *Rand) GetFrs(n int) ([]fr.Element, error) {
	out := make([]fr.Element, n)
	if rc := C.cdl_rand_get_frs(r.h, C.size_t(n), frPtr(out)); rc != 0 {
		return nil, errStatus(rc)
	}
	return out, nil
}

type statusError int32

func (e statusError) Error() string { return "curdle_b200 status " + itoa(int(e)) }
func errStatus(rc C.int32_t) error  { return statusError(rc) }
func itoa(v int) string {
	if v == 0 {
		return "0"
	}
	neg := v < 0
	if neg {
		v = -v
	}
	var b [20]byte
	i := len(b)
	for v > 0 {
		i--
		b[i] = byte('0' + v%10)
		v /= 10
	}
	if neg {
		i--
		b[i] = '-'
	}
	return string(b[i:])
}

// CRS is curdleproof.CRS (crs.go:10-18) resident on the device.
type CRS struct {
	h   *C.cdl_crs
	Ell int
}

// GenerateCRS is curdleproof.GenerateCRS(size, rand) (crs.go:20-59).
func (c *Context) GenerateCRS(size int, r *Rand) (*CRS, error) {
	var h *C.cdl_crs
	if rc := C.cdl_crs_generate(c.h, C.size_t(size), r.h, &h); rc != 0 {
		return nil, c.err(rc)
	}
	return &CRS{h, size}, nil
}

// CRSFromPoints uploads an existing CRS: Gs[ell] | Hs[4] | H | Gt | Gu | Gsum | Hsum.
func (c *Context) CRSFromPoints(ell int, pts []bls12381.G1Affine) (*CRS, error) {
	var h *C.cdl_crs
	if rc := C.cdl_crs_from_points(c.h, C.size_t(ell), affPtr(pts), &h); rc != 0 {
		return nil, c.err(rc)
	}
	return &CRS{h, ell}, nil
}

// Free releases the CRS.
func (s *CRS) Free() { C.cdl_crs_free(s.h) }

// Prove is curdleproof.Prove (curdleproof.go:38-197) followed by Proof.Serialize (:358-387); the
// caller decodes the bytes with Proof.FromReader (or keeps them: they are what goes on the wire).
func (c *Context) Prove(crs *CRS, Rs, Ss, Ts, Us []bls12381.G1Affine, M *bls12381.G1Jac, perm []uint32,
	k *fr.Element, rsM []fr.Element, r *Rand) ([]byte, error) {
	buf := make([]byte, 48*(18+10*32)+32*7+40)
	var n C.size_t
	rc := C.cdl_prove(c.h, crs.h, affPtr(Rs), affPtr(Ss), affPtr(Ts), affPtr(Us),
		(*C.cdl_g1_jac)(unsafe.Pointer(M)), (*C.uint32_t)(unsafe.Pointer(&perm[0])),
		(*C.cdl_fr)(unsafe.Pointer(k)), frPtr(rsM), r.h, (*C.uint8_t)(unsafe.Pointer(&buf[0])), C.size_t(len(buf)), &n)
	if rc != 0 {
		return nil, c.err(rc)
	}
	return buf[:n], nil
}

// SetBatchVerifyMin is cdl_set_batch_verify_min: lanes of at least proofs proofs check their whole batch
// with one combined MSM first (-1 = default, 0 = never).  Results do not depend on it.
func (c *Context) SetBatchVerifyMin(proofs int) error {
	if rc := C.cdl_set_batch_verify_min(c.h, C.int32_t(proofs)); rc != 0 {
		return c.err(rc)
	}
	return nil
}

// Verify is Proof.FromReader + curdleproof.Verify (curdleproof.go:199-318): (bool, error) as in the
// reference — (false, nil) for an invalid proof, (false, err) for malformed input.
func (c *Context) Verify(crs *CRS, proof []byte, Rs, Ss, Ts, Us []bls12381.G1Affine, M *bls12381.G1Jac, r *Rand) (bool, error) {
	var ok C.int32_t
	rc := C.cdl_verify(c.h, crs.h, (*C.uint8_t)(unsafe.Pointer(&proof[0])), C.size_t(len(proof)),
		affPtr(Rs), affPtr(Ss), affPtr(Ts), affPtr(Us), (*C.cdl_g1_jac)(unsafe.Pointer(M)), r.h, &ok)
	if rc != 0 {
		return false, c.err(rc)
	}
	return ok == 1, nil
}

// WhiskTracker / WhiskShuffleProofBytes cross as the byte arrays they already are
// (whisk/types.go:21-24,74-77): 96 bytes per tracker, 4576 bytes per proof.
const (
	TrackerSize      = C.CDL_WHISK_TRACKER_SIZE
	ShuffleProofSize = C.CDL_WHISK_SHUFFLE_PROOF_SIZE
)

// GenerateWhiskShuffleProofs is whisk.GenerateWhiskShuffleProof (whisk/whisk.go:63-114) for B
// independent instances in lock step: pre holds B*ell trackers, rands one generator per instance.
func (c *Context) GenerateWhiskShuffleProofs(crs *CRS, pre []byte, rands []*Rand) (post, proofs []byte, status []int32, err error) {
	B := len(rands)
	post = make([]byte, len(pre))
	proofs = make([]byte, B*ShuffleProofSize)
	status = make([]int32, B)
	hs := make([]*C.cdl_rand, B)
	for i, r := range rands {
		hs[i] = r.h
	}
	rc := C.cdl_whisk_generate_shuffle_proof_batch(c.h, crs.h, C.size_t(B), (*C.uint8_t)(unsafe.Pointer(&pre[0])),
		(**C.cdl_rand)(unsafe.Pointer(&hs[0])), (*C.uint8_t)(unsafe.Pointer(&post[0])),
		(*C.uint8_t)(unsafe.Pointer(&proofs[0])), C.size_t(ShuffleProofSize), (*C.int32_t)(unsafe.Pointer(&status[0])))
	if rc != 0 {
		err = c.err(rc)
	}
	return
}

// IsValidWhiskShuffleProofs is whisk.IsValidWhiskShuffleProof (whisk/whisk.go:20-61) for B instances:
// ok[b] is the reference's bool, status[b] != 0 its error.
func (c *Context) IsValidWhiskShuffleProofs(crs *CRS, pre, post, proofs []byte, rands []*Rand) (ok, status []int32, err error) {
	B := len(rands)
	ok = make([]int32, B)
	status = make([]int32, B)
	hs := make([]*C.cdl_rand, B)
	for i, r := range rands {
		hs[i] = r.h
	}
	rc := C.cdl_whisk_is_valid_shuffle_proof_batch(c.h, crs.h, C.size_t(B), (*C.uint8_t)(unsafe.Pointer(&pre[0])),
		(*C.uint8_t)(unsafe.Pointer(&post[0])), (*C.uint8_t)(unsafe.Pointer(&proofs[0])), C.size_t(ShuffleProofSize),
		(**C.cdl_rand)(unsafe.Pointer(&hs[0])), (*C.int32_t)(unsafe.Pointer(&ok[0])), (*C.int32_t)(unsafe.Pointer(&status[0])))
	if rc != 0 {
		err = c.err(rc)
	}
	return
}

// MatchWhiskTrackers finds which of the secrets ks own which of the trackers (96 bytes each): owner[t] is
// the smallest v with ks[v]·rG_t == krG_t, else -1; status[t] != 0 when tracker t does not decode
// (CDL_ERR_DECODE) or its rG is the point at infinity (CDL_ERR_PROTOCOL).  The reference leaves this
// check to the caller, one ScalarMultiplication per (key, tracker) pair.
func (c *Context) MatchWhiskTrackers(trackers []byte, ks []fr.Element) (owner, status []int32, err error) {
	if len(trackers) == 0 || len(trackers)%TrackerSize != 0 || len(ks) == 0 {
		return nil, nil, errStatus(C.int32_t(C.CDL_ERR_INVALID_ARG))
	}
	T := len(trackers) / TrackerSize
	owner = make([]int32, T)
	status = make([]int32, T)
	rc := C.cdl_whisk_match_trackers(c.h, C.size_t(T), (*C.uint8_t)(unsafe.Pointer(&trackers[0])), C.size_t(len(ks)),
		frPtr(ks), (*C.int32_t)(unsafe.Pointer(&owner[0])), (*C.int32_t)(unsafe.Pointer(&status[0])))
	if rc != 0 {
		return nil, nil, c.err(rc)
	}
	return owner, status, nil
}

// GenerateWhiskRegistrationBatch prepares the first-proposal Whisk registration of len(ks) validators: validator b
// draws r from rands[b] and gets the fresh tracker {r·G, k·r·G} (96 bytes), its k-commitment k·G (48 bytes) and
// the opening proof GenerateWhiskTrackerProof gives for them (128 bytes, one blinder drawn from rands[b] after
// r).  status[b] == CDL_ERR_PROTOCOL when r is 0 or 1 (rG at infinity or rG == G, which
// process_whisk_registration refuses); that validator draws no blinder and its bytes stay zero.  rands must hold
// one distinct *Rand per validator: the validators draw concurrently, so a Rand passed for two validators is a
// data race (a tool with one RNG for all validators draws into separate Rands, or seeds one per validator).
func (c *Context) GenerateWhiskRegistrationBatch(ks []fr.Element, rands []*Rand) (trackers, kComms, proofs []byte,
	status []int32, err error) {
	B := len(ks)
	if B == 0 || len(rands) != B {
		return nil, nil, nil, nil, errStatus(C.int32_t(C.CDL_ERR_INVALID_ARG))
	}
	trackers = make([]byte, B*TrackerSize)
	kComms = make([]byte, B*48)
	proofs = make([]byte, B*C.CDL_WHISK_TRACKER_PROOF_SIZE)
	status = make([]int32, B)
	rc := C.cdl_whisk_generate_registration_batch(c.h, C.size_t(B), frPtr(ks), randHandles(rands),
		(*C.uint8_t)(unsafe.Pointer(&trackers[0])), (*C.uint8_t)(unsafe.Pointer(&kComms[0])),
		(*C.uint8_t)(unsafe.Pointer(&proofs[0])), (*C.int32_t)(unsafe.Pointer(&status[0])))
	if rc != 0 {
		return nil, nil, nil, nil, c.err(rc)
	}
	return trackers, kComms, proofs, status, nil
}

func randHandles(rands []*Rand) **C.cdl_rand {
	hs := make([]*C.cdl_rand, len(rands))
	for i, r := range rands {
		hs[i] = r.h
	}
	return (**C.cdl_rand)(unsafe.Pointer(&hs[0]))
}

// ShufflePermuteCommitBatch is common.ShufflePermuteCommit (common/util.go:45-88) for B = len(rands) caller
// instances in lock step: Rs, Ss and perms hold B*ell entries (instance-major), ks one scalar per instance.
// status[b] is what the single call would return for instance b (CDL_ERR_INVALID_ARG for a permutation
// entry out of range, in which case rands[b] draws nothing).
func (c *Context) ShufflePermuteCommitBatch(crs *CRS, Rs, Ss []bls12381.G1Affine, perms []uint32, ks []fr.Element,
	rands []*Rand) (Ts, Us []bls12381.G1Affine, M []bls12381.G1Jac, rsM []fr.Element, status []int32, err error) {
	B := len(rands)
	if B == 0 || len(Rs) != B*crs.Ell || len(Ss) != B*crs.Ell || len(perms) != B*crs.Ell || len(ks) != B {
		return nil, nil, nil, nil, nil, errStatus(C.int32_t(C.CDL_ERR_INVALID_ARG))
	}
	Ts = make([]bls12381.G1Affine, len(Rs))
	Us = make([]bls12381.G1Affine, len(Rs))
	M = make([]bls12381.G1Jac, B)
	rsM = make([]fr.Element, 4*B)
	status = make([]int32, B)
	rc := C.cdl_shuffle_permute_commit_batch(c.h, crs.h, C.size_t(B), affPtr(Rs), affPtr(Ss),
		(*C.uint32_t)(unsafe.Pointer(&perms[0])), frPtr(ks), randHandles(rands), affPtr(Ts), affPtr(Us),
		(*C.cdl_g1_jac)(unsafe.Pointer(&M[0])), frPtr(rsM), (*C.int32_t)(unsafe.Pointer(&status[0])))
	if rc != 0 {
		return nil, nil, nil, nil, nil, c.err(rc)
	}
	return
}

// ProveBatch is curdleproof.Prove + Proof.Serialize for B = len(rands) caller instances in lock step (arrays
// as in ShufflePermuteCommitBatch, rsM 4 per instance).  proofs[b] is nil unless status[b] == 0.
func (c *Context) ProveBatch(crs *CRS, Rs, Ss, Ts, Us []bls12381.G1Affine, M []bls12381.G1Jac, perms []uint32,
	ks, rsM []fr.Element, rands []*Rand) (proofs [][]byte, status []int32, err error) {
	B := len(rands)
	n := B * crs.Ell
	if B == 0 || len(Rs) != n || len(Ss) != n || len(Ts) != n || len(Us) != n || len(M) != B || len(perms) != n ||
		len(ks) != B || len(rsM) != 4*B {
		return nil, nil, errStatus(C.int32_t(C.CDL_ERR_INVALID_ARG))
	}
	const proofCap = 48*(18+10*32) + 32*7 + 40
	buf := make([]byte, B*proofCap)
	lens := make([]C.size_t, B)
	status = make([]int32, B)
	rc := C.cdl_prove_batch(c.h, crs.h, C.size_t(B), affPtr(Rs), affPtr(Ss), affPtr(Ts), affPtr(Us),
		(*C.cdl_g1_jac)(unsafe.Pointer(&M[0])), (*C.uint32_t)(unsafe.Pointer(&perms[0])), frPtr(ks), frPtr(rsM),
		randHandles(rands), (*C.uint8_t)(unsafe.Pointer(&buf[0])), C.size_t(proofCap), &lens[0],
		(*C.int32_t)(unsafe.Pointer(&status[0])))
	if rc != 0 {
		return nil, nil, c.err(rc)
	}
	proofs = make([][]byte, B)
	for b := range proofs {
		if status[b] == 0 {
			proofs[b] = buf[b*proofCap : b*proofCap+int(lens[b])]
		}
	}
	return proofs, status, nil
}

// VerifyBatch is Proof.FromReader + curdleproof.Verify for B = len(rands) caller instances in lock step:
// ok[b] is the reference's bool and status[b] its error (what Verify would return for instance b).
func (c *Context) VerifyBatch(crs *CRS, proofs [][]byte, Rs, Ss, Ts, Us []bls12381.G1Affine, M []bls12381.G1Jac,
	rands []*Rand) (ok, status []int32, err error) {
	B := len(rands)
	n := B * crs.Ell
	if B == 0 || len(proofs) != B || len(Rs) != n || len(Ss) != n || len(Ts) != n || len(Us) != n || len(M) != B {
		return nil, nil, errStatus(C.int32_t(C.CDL_ERR_INVALID_ARG))
	}
	stride := 1
	for _, p := range proofs {
		if len(p) > stride {
			stride = len(p)
		}
	}
	buf := make([]byte, B*stride)
	lens := make([]C.size_t, B)
	for b, p := range proofs {
		copy(buf[b*stride:], p)
		lens[b] = C.size_t(len(p))
	}
	ok = make([]int32, B)
	status = make([]int32, B)
	rc := C.cdl_verify_batch(c.h, crs.h, C.size_t(B), (*C.uint8_t)(unsafe.Pointer(&buf[0])), C.size_t(stride), &lens[0],
		affPtr(Rs), affPtr(Ss), affPtr(Ts), affPtr(Us), (*C.cdl_g1_jac)(unsafe.Pointer(&M[0])), randHandles(rands),
		(*C.int32_t)(unsafe.Pointer(&ok[0])), (*C.int32_t)(unsafe.Pointer(&status[0])))
	if rc != 0 {
		return nil, nil, c.err(rc)
	}
	return ok, status, nil
}
