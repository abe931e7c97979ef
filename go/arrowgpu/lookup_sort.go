package arrowgpu

/*
#include "arrowgpu.h"
*/
import "C"

import (
	"context"
	"fmt"

	"github.com/apache/arrow-go/v18/arrow"
	"github.com/apache/arrow-go/v18/arrow/array"
	"github.com/apache/arrow-go/v18/arrow/compute"
	"github.com/apache/arrow-go/v18/arrow/compute/exec"
	"github.com/apache/arrow-go/v18/arrow/compute/internal/kernels"
	"github.com/apache/arrow-go/v18/arrow/memory"
)

// ---- is_in (scalar_set_lookup.go:70-171, kernels/scalar_set_lookup.go:112-413) ---------------------------------
//
// The reference's kernel state is a memo table of the value set; here it is the value set itself as ONE array of the
// argument's type (cast with SafeCastOptions and concatenated exactly where initSetLookup does it), and the table is
// built on the device inside ag_is_in.  Values are compared by their raw bytes on both sides, like the memo tables.

type setState struct {
	set      arrow.Array
	behavior C.int // NullMatchingBehavior: MATCH 0, SKIP 1, EMIT_NULL 2, INCONCLUSIVE 3 (= AG_NULL_*)
}

func initIsIn(ctx *exec.KernelCtx, args exec.KernelInitArgs) (exec.KernelState, error) {
	if args.Options == nil {
		return nil, fmt.Errorf("%w: calling a set lookup function without SetOptions", compute.ErrInvalid)
	}
	opts, ok := args.Options.(*compute.SetOptions)
	if !ok {
		return nil, fmt.Errorf("%w: expected SetOptions, got %T", compute.ErrInvalid, args.Options)
	}
	valueset, ok := opts.ValueSet.(compute.ArrayLikeDatum)
	if !ok {
		return nil, fmt.Errorf("%w: expected array-like datum, got %T", compute.ErrInvalid, opts.ValueSet)
	}
	argType := args.Inputs[0]
	var owned compute.Datum
	if !arrow.TypeEqual(valueset.Type(), argType) { // scalar_set_lookup.go:94-112: the set is cast to the argument's type
		result, err := compute.CastDatum(ctx.Ctx, valueset, compute.SafeCastOptions(argType))
		if err != nil {
			return nil, fmt.Errorf("%w: array type doesn't match type of values set: %s vs %s", compute.ErrInvalid, argType, valueset.Type())
		}
		owned = result
		valueset = result.(compute.ArrayLikeDatum)
	}
	if owned != nil {
		defer owned.Release()
	}
	var set arrow.Array
	switch valueset.Kind() {
	case compute.KindArray:
		set = valueset.(*compute.ArrayDatum).MakeArray()
	case compute.KindChunked:
		var err error
		if set, err = array.Concatenate(valueset.(*compute.ChunkedDatum).Value.Chunks(), exec.GetAllocator(ctx.Ctx)); err != nil {
			return nil, err
		}
	default:
		return nil, fmt.Errorf("%w: expected array or chunked array, got %s", compute.ErrInvalid, opts.ValueSet.Kind())
	}
	return &setState{set: set, behavior: C.int(opts.NullBehavior)}, nil
}

// isInExec writes the data and validity bitmaps of one batch (isInKernelExec :373-413).  The kernel is registered with
// CanWriteIntoSlices = false, so `out` is a fresh allocation at bit offset 0 — what the C entry point expects.
func isInExec(ctx *exec.KernelCtx, batch *exec.ExecSpan, out *exec.ExecResult) error {
	st := ctx.State.(*setState)
	in := &batch.Values[0].Array
	if out.Offset != 0 {
		return fmt.Errorf("%w: arrowgpu: is_in into a sliced output", arrow.ErrNotImplemented)
	}
	set := st.set.Data()
	var setValid *C.uint8_t
	if set.NullN() != 0 && set.Buffers()[0] != nil {
		setValid = bitmap(set.Buffers()[0].Bytes())
	}
	var setVals []byte
	if set.Len() > 0 {
		setVals = set.Buffers()[1].Bytes()
	}
	bw := in.Type.(arrow.FixedWidthDataType).BitWidth()
	var nulls C.int64_t
	err := check(C.ag_is_in(C.int(bw), base0(in.Buffers[1].Buf), validityOf(in), C.int64_t(in.Offset), C.int64_t(in.Len),
		base0(setVals), setValid, C.int64_t(set.Offset()), C.int64_t(set.Len()), st.behavior,
		bitmap(out.Buffers[1].Buf), bitmap(out.Buffers[0].Buf), &nulls))
	if err != nil {
		return err
	}
	out.Nulls = int64(nulls)
	return nil
}

func isInFunction() *compute.ScalarFunction {
	fn := compute.NewScalarFunction("is_in", compute.Unary(), compute.EmptyFuncDoc)
	for _, ty := range numericTypes {
		kn := exec.NewScalarKernel([]exec.InputType{exec.NewExactInput(ty)}, exec.NewOutputType(arrow.FixedWidthTypes.Boolean), isInExec, initIsIn)
		kn.MemAlloc = exec.MemPrealloc                 // scalar_set_lookup.go:190-191
		kn.NullHandling = exec.NullComputedPrealloc
		kn.CanWriteIntoSlices = false
		kn.CleanupFn = func(state exec.KernelState) error {
			if s, ok := state.(*setState); ok && s.set != nil {
				s.set.Release()
				s.set = nil
			}
			return nil
		}
		if err := fn.AddKernel(kn); err != nil {
			panic(err)
		}
	}
	return fn
}

// ---- unique (vector_hash.go:105-113, kernels/vector_hash.go) -------------------------------------------------------
//
// The reference hashes chunk by chunk into one memo table and materialises it in Finalize; ag_unique needs the whole
// column at once (the first row of every key is a global minimum), so the kernel is not chunk-wise: a chunked input is
// concatenated first.  Output: the distinct values in order of first appearance, one null where it first appears.

func uniqueExec(ctx *exec.KernelCtx, batch *exec.ExecSpan, out *exec.ExecResult) error {
	in := &batch.Values[0].Array
	bw := in.Type.(arrow.FixedWidthDataType).BitWidth()
	preallocate(ctx, in.Len, bw, in.MayHaveNulls(), out) // n slots are always enough; Len is trimmed below
	var outLen, outNulls C.int64_t
	err := check(C.ag_unique(C.int(bw), base0(in.Buffers[1].Buf), validityOf(in), C.int64_t(in.Offset), C.int64_t(in.Len),
		base0(out.Buffers[1].Buf), bitmap(out.Buffers[0].Buf), &outLen, &outNulls))
	if err != nil {
		return err
	}
	out.Len, out.Nulls = int64(outLen), int64(outNulls)
	return nil
}

func uniqueChunked(ctx *exec.KernelCtx, cols []*arrow.Chunked, out *exec.ExecResult) ([]*exec.ExecResult, error) {
	arr, err := array.Concatenate(cols[0].Chunks(), exec.GetAllocator(ctx.Ctx))
	if err != nil {
		return nil, err
	}
	defer arr.Release()
	span := exec.ExecSpan{Len: int64(arr.Len()), Values: make([]exec.ExecValue, 1)}
	span.Values[0].Array.SetMembers(arr.Data())
	if err := uniqueExec(ctx, &span, out); err != nil {
		return nil, err
	}
	return []*exec.ExecResult{out}, nil
}

func uniqueFunction() *compute.VectorFunction {
	fn := compute.NewVectorFunction("unique", compute.Unary(), compute.EmptyFuncDoc)
	for _, ty := range numericTypes {
		k := exec.NewVectorKernel([]exec.InputType{exec.NewExactInput(ty)}, kernels.OutputFirstType, uniqueExec, nil)
		k.CanExecuteChunkWise = false
		k.ExecChunked = uniqueChunked
		k.NullHandling = exec.NullComputedNoPrealloc
		k.MemAlloc = exec.MemNoPrealloc
		if err := fn.AddKernel(k); err != nil {
			panic(err)
		}
	}
	return fn
}

// ---- sort_indices (vector_sort.go:42-204, kernels.SortIndices vector_sort.go:385-481) -------------------------------
//
// A MetaFunction in the reference.  The GPU entry sorts ONE contiguous fixed-width column (stable, NaNs after the finite
// values, nulls per NullPlacement); chunked inputs, record batches, tables and multi-key sorts go to the parent's
// implementation, like every other shape this package does not cover.

func sortIndicesFunction(parent compute.Function) *compute.MetaFunction {
	return compute.NewMetaFunction("sort_indices", compute.Unary(), compute.EmptyFuncDoc,
		func(ctx context.Context, opts compute.FunctionOptions, args ...compute.Datum) (compute.Datum, error) {
			keys, isKeys := opts.(compute.SortOptions)
			if in, ok := args[0].(*compute.ArrayDatum); ok && isKeys && len(keys) >= 1 && isNumeric(in.Type()) {
				return sortOneColumn(ctx, in.Value, keys[0]) // a bare array uses the first key only (vector_sort.go:138-142)
			}
			if parent == nil {
				return nil, fmt.Errorf("%w: unsupported type for sort_indices operation: %s", arrow.ErrNotImplemented, args[0])
			}
			return parent.Execute(ctx, opts, args...)
		})
}

func isNumeric(dt arrow.DataType) bool {
	for _, ty := range numericTypes {
		if arrow.TypeEqual(ty, dt) {
			return true
		}
	}
	return false
}

func sortOneColumn(ctx context.Context, col arrow.ArrayData, key compute.SortKey) (compute.Datum, error) {
	n := col.Len()
	buf := memory.NewResizableBuffer(exec.GetAllocator(ctx))
	buf.Resize(n * 8)
	var vals []byte
	if n > 0 {
		vals = col.Buffers()[1].Bytes()
	}
	var valid *C.uint8_t
	if col.NullN() != 0 && col.Buffers()[0] != nil {
		valid = bitmap(col.Buffers()[0].Bytes())
	}
	var nulls, nans C.int64_t
	// arrow.Type ids are the AG_TYPE_* ids; SortOrder / NullPlacement are 0 / 1 on both sides (kernels/vector_sort.go:34-46)
	err := check(C.ag_sort_indices(C.int(col.DataType().ID()), base0(vals), valid, C.int64_t(col.Offset()), C.int64_t(n),
		C.int(key.Order), C.int(key.NullPlacement), (*C.uint64_t)(base0(buf.Bytes())), &nulls, &nans))
	if err != nil {
		buf.Release()
		return nil, err
	}
	out := array.NewData(arrow.PrimitiveTypes.Uint64, n, []*memory.Buffer{nil, buf}, nil, 0, 0)
	buf.Release() // NewData retained it
	return &compute.ArrayDatum{Value: out}, nil
}

// ---- dictionary_encode (vector_hash.go:105-125, kernels/vector_hash.go:83-241,359-385,854-925) -----------------------
//
// Like unique, ag_dictionary_encode needs the whole column at once (a value's dictionary position is the rank of its
// first row), so the kernel is not chunk-wise: a chunked input is concatenated, encoded in one call, and its indices are
// split back into the input's chunk lengths.  The dictionary waits in the kernel state until Finalize attaches it to
// every result (dictionaryEncodeFinalize :854-872), so all chunks share one dictionary.  Dictionary inputs (the
// identity kernel) and every non-numeric type go to the parent registry.

type dictEncodeState struct {
	nullEncoding C.int // NullEncodingMask 0 / NullEncodingEncode 1 (= AG_NULL_ENCODING_*)
	dict         arrow.ArrayData
}

// initDictEncode restates parseDictionaryEncodeOptions (kernels/vector_hash.go:811-829).
func initDictEncode(_ *exec.KernelCtx, args exec.KernelInitArgs) (exec.KernelState, error) {
	opts := compute.DictionaryEncodeOptions{}
	switch o := args.Options.(type) {
	case nil:
	case compute.DictionaryEncodeOptions:
		opts = o
	case *compute.DictionaryEncodeOptions:
		if o != nil {
			opts = *o
		}
	default:
		return nil, fmt.Errorf("%w: expected DictionaryEncodeOptions, got %T", arrow.ErrInvalid, args.Options)
	}
	if opts.NullEncoding != compute.NullEncodingMask && opts.NullEncoding != compute.NullEncodingEncode {
		return nil, fmt.Errorf("%w: invalid null encoding behavior %d", arrow.ErrInvalid, opts.NullEncoding)
	}
	return &dictEncodeState{nullEncoding: C.int(opts.NullEncoding)}, nil
}

func dictEncodeExec(ctx *exec.KernelCtx, batch *exec.ExecSpan, out *exec.ExecResult) error {
	st := ctx.State.(*dictEncodeState)
	in := &batch.Values[0].Array
	bw := in.Type.(arrow.FixedWidthDataType).BitWidth()
	mask := st.nullEncoding == C.AG_NULL_ENCODING_MASK
	preallocate(ctx, in.Len, 32, in.MayHaveNulls() && mask, out)
	dictVals := ctx.Allocate(int(in.Len) * (bw / 8)) // n entries are always enough; the length is trimmed below
	var dictValid *memory.Buffer
	var dictValidBytes []byte
	if in.MayHaveNulls() && !mask {
		dictValid = ctx.AllocateBitmap(in.Len)
		dictValidBytes = dictValid.Bytes()
	}
	var dictLen, nulls C.int64_t
	err := check(C.ag_dictionary_encode(C.int(bw), base0(in.Buffers[1].Buf), validityOf(in), C.int64_t(in.Offset), C.int64_t(in.Len),
		st.nullEncoding, (*C.int32_t)(base0(out.Buffers[1].Buf)), bitmap(out.Buffers[0].Buf), base0(dictVals.Bytes()), bitmap(dictValidBytes),
		&dictLen, &nulls))
	if err != nil {
		dictVals.Release()
		if dictValid != nil {
			dictValid.Release()
		}
		return err
	}
	out.Nulls = int64(nulls)
	dictNulls := 0
	if dictValid != nil {
		dictNulls = array.UnknownNullCount
	}
	if st.dict != nil {
		st.dict.Release()
	}
	st.dict = array.NewData(in.Type, int(dictLen), []*memory.Buffer{dictValid, dictVals}, nil, dictNulls, 0)
	dictVals.Release() // NewData retained them
	if dictValid != nil {
		dictValid.Release()
	}
	return nil
}

func dictEncodeChunked(ctx *exec.KernelCtx, cols []*arrow.Chunked, out *exec.ExecResult) ([]*exec.ExecResult, error) {
	arr, err := array.Concatenate(cols[0].Chunks(), exec.GetAllocator(ctx.Ctx))
	if err != nil {
		return nil, err
	}
	defer arr.Release()
	span := exec.ExecSpan{Len: int64(arr.Len()), Values: make([]exec.ExecValue, 1)}
	span.Values[0].Array.SetMembers(arr.Data())
	if err := dictEncodeExec(ctx, &span, out); err != nil {
		return nil, err
	}
	whole := out.MakeData()
	defer whole.Release()
	out.Release() // the chunks below hold their own references
	results := make([]*exec.ExecResult, 0, len(cols[0].Chunks()))
	pos := int64(0)
	for _, ch := range cols[0].Chunks() {
		part := array.NewSliceData(whole, pos, pos+int64(ch.Len()))
		r := &exec.ExecResult{}
		r.TakeOwnership(part)
		part.Release()
		results = append(results, r)
		pos += int64(ch.Len())
	}
	return results, nil
}

func dictEncodeFinalize(ctx *exec.KernelCtx, results []*exec.ArraySpan) ([]*exec.ArraySpan, error) {
	st := ctx.State.(*dictEncodeState)
	if st.dict == nil {
		return results, nil
	}
	for _, r := range results {
		var d exec.ArraySpan
		d.TakeOwnership(st.dict)
		r.SetDictionary(&d)
	}
	st.dict.Release()
	st.dict = nil
	return results, nil
}

func dictEncodeFunction() *compute.VectorFunction {
	fn := compute.NewVectorFunction("dictionary_encode", compute.Unary(), compute.EmptyFuncDoc)
	outType := exec.NewComputedOutputType(func(_ *exec.KernelCtx, args []arrow.DataType) (arrow.DataType, error) {
		return &arrow.DictionaryType{IndexType: arrow.PrimitiveTypes.Int32, ValueType: args[0]}, nil
	})
	for _, ty := range numericTypes {
		k := exec.NewVectorKernel([]exec.InputType{exec.NewExactInput(ty)}, outType, dictEncodeExec, initDictEncode)
		k.CanExecuteChunkWise = false
		k.OutputChunked = true
		k.ExecChunked = dictEncodeChunked
		k.Finalize = dictEncodeFinalize
		k.NullHandling = exec.NullComputedNoPrealloc
		k.MemAlloc = exec.MemNoPrealloc
		if err := fn.AddKernel(k); err != nil {
			panic(err)
		}
	}
	return fn
}

// registerLookupSort adds is_in, unique, dictionary_encode and sort_indices to a registry built by NewRegistry.
func registerLookupSort(reg, parent compute.FunctionRegistry) {
	addScalar(reg, parent, isInFunction())
	addVector(reg, parent, uniqueFunction())
	addVector(reg, parent, dictEncodeFunction())
	p, _ := parent.GetFunction("sort_indices")
	reg.AddFunction(sortIndicesFunction(p), true)
}
