// Package gpu binds libcurdle_b200.so (include/curdle_b200.h) for go-curdleproofs.
//
// Drop this directory into the reference as `gpu/` (module path
// github.com/jsign/curdleproofs/gpu), point CGO at the header and the shared library (the
// #cgo lines below assume third_party/curdle_b200/{include,lib}), and replace the gnark-crypto
// call sites listed in INTEGRATION.md §2 with the methods of *Context.  gnark's G1Affine /
// G1Jac / fr.Element are plain value arrays with exactly the layout the header documents
// (6x64 / 4x64 little-endian Montgomery limbs), so Go slices cross with unsafe.Pointer(&s[0])
// and the library keeps no Go pointer after a call returns (cgo pointer rule).
//
// There is no CPU fallback: New fails when no CUDA device is present.
//
// NOTE: committed without having been compiled (no Go toolchain in the build image or on the
// GPU box); every C entry point used here is exercised through the same ABI by the ctypes
// tests (tests/test_gpu_*.py).
package gpu

/*
#cgo CFLAGS: -I${SRCDIR}/../third_party/curdle_b200/include
#cgo LDFLAGS: -L${SRCDIR}/../third_party/curdle_b200/lib -lcurdle_b200
#include <stdlib.h>
#include "curdle_b200.h"
*/
import "C"

import (
	"errors"
	"fmt"
	"unsafe"

	bls12381 "github.com/consensys/gnark-crypto/ecc/bls12-381"
	"github.com/consensys/gnark-crypto/ecc/bls12-381/fr"
)

// Context is one device + stream (or a list of devices, NewDevices); safe for concurrent use (calls
// serialise on the context).
type Context struct{ h *C.cdl_ctx }

// New opens CUDA device `device`.
func New(device int) (*Context, error) {
	var h *C.cdl_ctx
	if rc := C.cdl_create(C.int(device), &h); rc != 0 {
		return nil, fmt.Errorf("cdl_create: status %d (no CPU fallback)", int(rc))
	}
	return &Context{h}, nil
}

// NewDevices opens one context over the CUDA devices listed (at most 16; a device may appear more
// than once).  Its batched calls (Whisk shuffle and tracker proofs, the curdleproof batches, tracker
// matching) are dealt to the devices in contiguous blocks; everything else runs on devices[0].
// Results do not depend on the list.  A multi-GPU node uses one such context instead of a process
// per GPU.
func NewDevices(devices []int) (*Context, error) {
	if len(devices) == 0 {
		return nil, errors.New("NewDevices: empty device list")
	}
	ids := make([]C.int32_t, len(devices))
	for i, d := range devices {
		ids[i] = C.int32_t(d)
	}
	var h *C.cdl_ctx
	if rc := C.cdl_create_devices(&ids[0], C.size_t(len(ids)), &h); rc != 0 {
		return nil, fmt.Errorf("cdl_create_devices: status %d (no CPU fallback)", int(rc))
	}
	return &Context{h}, nil
}

// Devices returns the context's device list (one entry per device slot).
func (c *Context) Devices() ([]int, error) {
	var n C.size_t
	if rc := C.cdl_context_devices(c.h, nil, 0, &n); rc != 0 {
		return nil, c.err(rc)
	}
	ids := make([]C.int32_t, n)
	if n > 0 {
		if rc := C.cdl_context_devices(c.h, &ids[0], n, &n); rc != 0 {
			return nil, c.err(rc)
		}
	}
	out := make([]int, len(ids))
	for i, d := range ids {
		out[i] = int(d)
	}
	return out, nil
}

// Close releases the device resources of the context.
func (c *Context) Close() { C.cdl_destroy(c.h) }

func (c *Context) err(rc C.int32_t) error {
	return fmt.Errorf("curdle_b200 %d: %s", int(rc), C.GoString(C.cdl_last_error(c.h)))
}

func affPtr(s []bls12381.G1Affine) *C.cdl_g1_affine {
	if len(s) == 0 {
		return nil
	}
	return (*C.cdl_g1_affine)(unsafe.Pointer(&s[0]))
}

func frPtr(s []fr.Element) *C.cdl_fr {
	if len(s) == 0 {
		return nil
	}
	return (*C.cdl_fr)(unsafe.Pointer(&s[0]))
}

// MultiExp replaces (*G1Jac).MultiExp(points, scalars, common.MultiExpConf) at all 39 call
// sites (curdleproof.go:72,75,109,113; msmaccumulator/msmaccumulator.go:59; ...).
func (c *Context) MultiExp(points []bls12381.G1Affine, scalars []fr.Element) (bls12381.G1Jac, error) {
	var out bls12381.G1Jac
	if len(points) != len(scalars) {
		return out, errors.New("len(points) != len(scalars)") // gnark's only MultiExp error
	}
	if rc := C.cdl_g1_msm(c.h, affPtr(points), frPtr(scalars), C.size_t(len(points)),
		(*C.cdl_g1_jac)(unsafe.Pointer(&out))); rc != 0 {
		return out, c.err(rc)
	}
	return out, nil
}

// MultiExpBatch runs k independent MSMs in one launch: MSM j covers
// points/scalars[offsets[j]:offsets[j+1]] (the 4 / 6 MSMs of one IPA / SameMSM round,
// innerproductargument.go:108-138, samemultiscalarargument.go:93-111).  Affine results.
func (c *Context) MultiExpBatch(points []bls12381.G1Affine, scalars []fr.Element, offsets []uint32) ([]bls12381.G1Affine, error) {
	k := len(offsets) - 1
	if k <= 0 {
		return nil, nil
	}
	out := make([]bls12381.G1Affine, k)
	if rc := C.cdl_g1_msm_batch(c.h, affPtr(points), frPtr(scalars), (*C.uint32_t)(unsafe.Pointer(&offsets[0])),
		C.size_t(k), affPtr(out)); rc != 0 {
		return nil, c.err(rc)
	}
	return out, nil
}

// Fold replaces the serial loops L[i].Add(&L[i], tmp.ScalarMultiplication(&R[i], x))
// (innerproductargument.go:155-166, samemultiscalarargument.go:129-135): L[i] += x*R[i] in place.
func (c *Context) Fold(L, R []bls12381.G1Affine, x *fr.Element) error {
	if len(L) != len(R) {
		return errors.New("len(L) != len(R)")
	}
	if rc := C.cdl_g1_fold(c.h, affPtr(L), affPtr(R), (*C.cdl_fr)(unsafe.Pointer(x)), C.size_t(len(L))); rc != 0 {
		return c.err(rc)
	}
	return nil
}

// ScalarMulBatch replaces loops of G1Affine.ScalarMultiplication (common/util.go:55-63,
// grandproductargument.go:94-103); a single scalar (len(s) == 1) is broadcast.
func (c *Context) ScalarMulBatch(in []bls12381.G1Affine, s []fr.Element) ([]bls12381.G1Affine, error) {
	out := make([]bls12381.G1Affine, len(in))
	stride := C.size_t(1)
	if len(s) == 1 {
		stride = 0
	} else if len(s) != len(in) {
		return nil, errors.New("len(s) must be 1 or len(in)")
	}
	if rc := C.cdl_g1_scalar_mul_affine(c.h, affPtr(in), frPtr(s), C.size_t(len(in)), stride, affPtr(out)); rc != 0 {
		return nil, c.err(rc)
	}
	return out, nil
}

// BatchScalarMultiplicationG1 replaces bls12381.BatchScalarMultiplicationG1: scalars[i] * base for one base
// in G1 and many scalars (k-commitments kG, initial trackers (G, kG), blinder products r*G).  A base outside
// G1 is an error.  The context caches the fixed-base tables of its four most recently used bases.
func (c *Context) BatchScalarMultiplicationG1(base *bls12381.G1Affine, scalars []fr.Element) ([]bls12381.G1Affine, error) {
	out := make([]bls12381.G1Affine, len(scalars))
	if len(scalars) == 0 {
		return out, nil
	}
	if rc := C.cdl_g1_batch_scalar_mul_base(c.h, (*C.cdl_g1_affine)(unsafe.Pointer(base)), frPtr(scalars),
		C.size_t(len(scalars)), affPtr(out), nil); rc != 0 {
		return nil, c.err(rc)
	}
	return out, nil
}

// BatchScalarMultiplicationG1Compressed is BatchScalarMultiplicationG1 returning the 48-byte compressed
// encodings (G1Affine.Bytes()) of the products, len(scalars) * 48 bytes: the k-commitments kG of many
// validators, or the krG halves of their trackers.
func (c *Context) BatchScalarMultiplicationG1Compressed(base *bls12381.G1Affine, scalars []fr.Element) ([]byte, error) {
	out := make([]byte, 48*len(scalars))
	if len(scalars) == 0 {
		return out, nil
	}
	if rc := C.cdl_g1_batch_scalar_mul_base(c.h, (*C.cdl_g1_affine)(unsafe.Pointer(base)), frPtr(scalars),
		C.size_t(len(scalars)), nil, (*C.uint8_t)(unsafe.Pointer(&out[0]))); rc != 0 {
		return nil, c.err(rc)
	}
	return out, nil
}

// BatchJacobianToAffine replaces bls12381.BatchJacobianToAffineG1 (transcript/transcript.go:26).
func (c *Context) BatchJacobianToAffine(in []bls12381.G1Jac) ([]bls12381.G1Affine, error) {
	out := make([]bls12381.G1Affine, len(in))
	if len(in) == 0 {
		return out, nil
	}
	if rc := C.cdl_g1_batch_to_affine(c.h, (*C.cdl_g1_jac)(unsafe.Pointer(&in[0])), C.size_t(len(in)), affPtr(out)); rc != 0 {
		return nil, c.err(rc)
	}
	return out, nil
}

// SumAffine replaces the Gsum / Hsum loops of crs.go:41-48.
func (c *Context) SumAffine(in []bls12381.G1Affine) (bls12381.G1Affine, error) {
	var out bls12381.G1Affine
	if rc := C.cdl_g1_sum_affine(c.h, affPtr(in), C.size_t(len(in)), (*C.cdl_g1_affine)(unsafe.Pointer(&out))); rc != 0 {
		return out, c.err(rc)
	}
	return out, nil
}

// Compress replaces G1Affine.Bytes() over a list (whisk/types.go:79-84): 48 bytes per point.
func (c *Context) Compress(in []bls12381.G1Affine) ([]byte, error) {
	out := make([]byte, 48*len(in))
	if len(in) == 0 {
		return out, nil
	}
	if rc := C.cdl_g1_compress(c.h, affPtr(in), C.size_t(len(in)), (*C.uint8_t)(unsafe.Pointer(&out[0]))); rc != 0 {
		return nil, c.err(rc)
	}
	return out, nil
}

// Decompress replaces G1Affine.SetBytes (curve + subgroup checks) over n 48-byte encodings
// (whisk/types.go:86-95).  status[i] != 0 names the reason point i was rejected.
func (c *Context) Decompress(enc []byte) (pts []bls12381.G1Affine, status []byte, err error) {
	n := len(enc) / 48
	pts = make([]bls12381.G1Affine, n)
	status = make([]byte, n)
	if n == 0 {
		return
	}
	rc := C.cdl_g1_decompress(c.h, (*C.uint8_t)(unsafe.Pointer(&enc[0])), C.size_t(n), affPtr(pts),
		(*C.uint8_t)(unsafe.Pointer(&status[0])))
	if rc != 0 {
		err = c.err(rc)
	}
	return
}
