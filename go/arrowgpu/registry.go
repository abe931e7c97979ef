package arrowgpu

/*
#include "arrowgpu.h"
*/
import "C"

import (
	"context"

	"github.com/apache/arrow-go/v18/arrow"
	"github.com/apache/arrow-go/v18/arrow/compute"
	"github.com/apache/arrow-go/v18/arrow/compute/exec"
	"github.com/apache/arrow-go/v18/arrow/compute/internal/kernels"
)

// The ten numeric types of the reference's arithmetic / comparison kernel lists (scalar_arithmetic.go:86-95,
// scalar_comparisons.go:654-716).
var numericTypes = []arrow.DataType{
	arrow.PrimitiveTypes.Int8, arrow.PrimitiveTypes.Uint8, arrow.PrimitiveTypes.Int16, arrow.PrimitiveTypes.Uint16,
	arrow.PrimitiveTypes.Int32, arrow.PrimitiveTypes.Uint32, arrow.PrimitiveTypes.Int64, arrow.PrimitiveTypes.Uint64,
	arrow.PrimitiveTypes.Float32, arrow.PrimitiveTypes.Float64,
}

// intTypes of the reference's bitwise / shift kernel lists (scalar_arithmetic.go:245-255,401-412)
var integerTypes = numericTypes[:8]

// delegating is a compute.Function that runs the GPU ScalarFunction when its kernels match the argument types exactly
// and hands every other call (promotions, decimals, temporal types, dictionary inputs ...) to the function of the same
// name in the parent registry.  This is forced by the reference: dispatch is first-match over an unexported kernel
// slice (functions.go:209-213), and the built-ins' promotion lives in unexported wrappers whose Execute passes the
// wrapper to the unexported execInternal (arithmetic.go:92-140) — an external ScalarFunction gets exact dispatch only
// (functions.go:260-262).
type delegating struct {
	*compute.ScalarFunction
	parent compute.Function
}

func (d *delegating) Execute(ctx context.Context, opts compute.FunctionOptions, args ...compute.Datum) (compute.Datum, error) {
	types := make([]arrow.DataType, len(args))
	for i, a := range args {
		types[i] = a.(compute.ArrayLikeDatum).Type()
	}
	if _, err := d.ScalarFunction.DispatchExact(types...); err == nil {
		return d.ScalarFunction.Execute(ctx, opts, args...)
	}
	if d.parent != nil {
		return d.parent.Execute(ctx, opts, args...)
	}
	return d.ScalarFunction.Execute(ctx, opts, args...) // reports the dispatch error
}

func (d *delegating) DispatchBest(vals ...arrow.DataType) (exec.Kernel, error) {
	if k, err := d.ScalarFunction.DispatchExact(vals...); err == nil {
		return k, nil
	}
	if d.parent != nil {
		return d.parent.DispatchBest(vals...)
	}
	return d.ScalarFunction.DispatchBest(vals...)
}

func addScalar(reg, parent compute.FunctionRegistry, fn *compute.ScalarFunction) {
	p, _ := parent.GetFunction(fn.Name())
	reg.AddFunction(&delegating{ScalarFunction: fn, parent: p}, true)
}

func binaryKernel(ty arrow.DataType, out arrow.DataType, ex exec.ArrayKernelExec, nulls exec.NullHandling) exec.ScalarKernel {
	k := exec.NewScalarKernel([]exec.InputType{exec.NewExactInput(ty), exec.NewExactInput(ty)}, exec.NewOutputType(out), ex, nil)
	k.NullHandling = nulls
	return k
}

// NewRegistry returns a child of the global registry (registry.go:69) whose entries shadow the built-ins
// (GetFunction looks in the child first, :120-133).  Select it per call:
//
//	ctx = compute.SetExecCtx(ctx, compute.ExecCtx{Registry: arrowgpu.NewRegistry(), ChunkSize: math.MaxInt64, PreallocContiguous: true})
//	out, err := compute.Add(ctx, compute.ArithmeticOptions{}, left, right)
func NewRegistry() compute.FunctionRegistry {
	parent := compute.GetFunctionRegistry()
	reg := compute.NewChildRegistry(parent)

	// ---- add / sub(tract) / multiply (+ _unchecked): base_arithmetic_amd64.go:67-152 picks the native loop for the
	// unchecked ops and for floats; integral checked ops go through ScalarBinaryNotNull (:103-106)
	for _, f := range []struct {
		names   []string
		op      C.int8_t
		checked bool
	}{
		{[]string{"add"}, C.AG_OP_ADD_CHECKED, true}, {[]string{"add_unchecked"}, C.AG_OP_ADD, false},
		{[]string{"sub", "subtract"}, C.AG_OP_SUB_CHECKED, true}, {[]string{"sub_unchecked", "subtract_unchecked"}, C.AG_OP_SUB, false},
		{[]string{"multiply"}, C.AG_OP_MUL_CHECKED, true}, {[]string{"multiply_unchecked"}, C.AG_OP_MUL, false},
	} {
		for _, name := range f.names {
			fn := compute.NewScalarFunction(name, compute.Binary(), compute.EmptyFuncDoc)
			for _, ty := range numericTypes {
				ex := arithExec(f.op)
				if f.checked && arrow.IsInteger(ty.ID()) {
					ex = checkedExec(f.op)
				}
				if err := fn.AddKernel(binaryKernel(ty, ty, ex, exec.NullIntersection)); err != nil {
					panic(err)
				}
			}
			addScalar(reg, parent, fn)
		}
	}
	// ---- divide / divide_unchecked: every kernel is ScalarBinaryNotNull (base_arithmetic.go:154-161,287-294 integers —
	// a zero divisor fails in BOTH flavours —, :386-397 floats — only the checked one fails)
	for name, op := range map[string]C.int8_t{"divide": C.AG_OP_DIV_CHECKED, "divide_unchecked": C.AG_OP_DIV} {
		fn := compute.NewScalarFunction(name, compute.Binary(), compute.EmptyFuncDoc)
		for _, ty := range numericTypes {
			if err := fn.AddKernel(binaryKernel(ty, ty, checkedExec(op), exec.NullIntersection)); err != nil {
				panic(err)
			}
		}
		addScalar(reg, parent, fn)
	}
	// ---- bit_wise_and / or / xor (every slot, like the arithmetic loops) and bit_wise_not (arithmetic.go:944-972)
	for name, op := range map[string]C.int8_t{"bit_wise_and": C.AG_OP_BIT_AND, "bit_wise_or": C.AG_OP_BIT_OR, "bit_wise_xor": C.AG_OP_BIT_XOR} {
		fn := compute.NewScalarFunction(name, compute.Binary(), compute.EmptyFuncDoc)
		for _, ty := range integerTypes {
			if err := fn.AddKernel(binaryKernel(ty, ty, arithExec(op), exec.NullIntersection)); err != nil {
				panic(err)
			}
		}
		addScalar(reg, parent, fn)
	}
	{
		fn := compute.NewScalarFunction("bit_wise_not", compute.Unary(), compute.EmptyFuncDoc)
		for _, ty := range integerTypes {
			k := exec.NewScalarKernel([]exec.InputType{exec.NewExactInput(ty)}, exec.NewOutputType(ty), unaryExec(C.AG_OP_BIT_NOT), nil)
			if err := fn.AddKernel(k); err != nil {
				panic(err)
			}
		}
		addScalar(reg, parent, fn)
	}
	// ---- shift_left / shift_right (+ _unchecked), arithmetic.go:974-996, kernels scalar_arithmetic.go:293-412
	for name, op := range map[string]C.int8_t{"shift_left": C.AG_OP_SHIFT_LEFT_CHECKED, "shift_left_unchecked": C.AG_OP_SHIFT_LEFT,
		"shift_right": C.AG_OP_SHIFT_RIGHT_CHECKED, "shift_right_unchecked": C.AG_OP_SHIFT_RIGHT} {
		fn := compute.NewScalarFunction(name, compute.Binary(), compute.EmptyFuncDoc)
		for _, ty := range integerTypes {
			if err := fn.AddKernel(binaryKernel(ty, ty, checkedExec(op), exec.NullIntersection)); err != nil { // errShift worded by the library
				panic(err)
			}
		}
		addScalar(reg, parent, fn)
	}
	// ---- abs / negate (+ _unchecked) and sign
	for name, op := range map[string]C.int8_t{"abs": C.AG_OP_ABS_CHECKED, "abs_unchecked": C.AG_OP_ABS, "negate": C.AG_OP_NEGATE_CHECKED, "negate_unchecked": C.AG_OP_NEGATE, "sign": C.AG_OP_SIGN} {
		fn := compute.NewScalarFunction(name, compute.Unary(), compute.EmptyFuncDoc)
		for _, ty := range numericTypes {
			out := ty
			if name == "sign" && arrow.IsInteger(ty.ID()) {
				out = arrow.PrimitiveTypes.Int8 // base_arithmetic.go:398-442
				if arrow.IsUnsignedInteger(ty.ID()) {
					out = arrow.PrimitiveTypes.Uint8
				}
			}
			k := exec.NewScalarKernel([]exec.InputType{exec.NewExactInput(ty)}, exec.NewOutputType(out), unaryExec(op), nil)
			if err := fn.AddKernel(k); err != nil {
				panic(err)
			}
		}
		addScalar(reg, parent, fn)
	}
	// ---- comparisons -> boolean (scalar_compare.go:102-153); LT / LE are the flipped GT / GE
	for name, cmp := range map[string]C.int{"equal": C.AG_CMP_EQ, "not_equal": C.AG_CMP_NE, "greater": C.AG_CMP_GT,
		"greater_equal": C.AG_CMP_GE, "less": C.AG_CMP_LT, "less_equal": C.AG_CMP_LE} {
		fn := compute.NewScalarFunction(name, compute.Binary(), compute.EmptyFuncDoc)
		for _, ty := range numericTypes {
			if err := fn.AddKernel(binaryKernel(ty, arrow.FixedWidthTypes.Boolean, compareExec(cmp), exec.NullIntersection)); err != nil {
				panic(err)
			}
		}
		addScalar(reg, parent, fn)
	}
	// ---- boolean and Kleene kernels (scalar_bool.go:123-140)
	b := arrow.FixedWidthTypes.Boolean
	for name, op := range map[string]C.int{"and": C.AG_BITOP_AND, "or": C.AG_BITOP_OR, "xor": C.AG_BITOP_XOR, "and_not": C.AG_BITOP_ANDNOT} {
		fn := compute.NewScalarFunction(name, compute.Binary(), compute.EmptyFuncDoc)
		if err := fn.AddKernel(binaryKernel(b, b, bitmapOpExec(op), exec.NullIntersection)); err != nil {
			panic(err)
		}
		addScalar(reg, parent, fn)
	}
	for name, op := range map[string]C.int{"and_kleene": C.AG_KLEENE_AND, "or_kleene": C.AG_KLEENE_OR, "and_not_kleene": C.AG_KLEENE_ANDNOT} {
		fn := compute.NewScalarFunction(name, compute.Binary(), compute.EmptyFuncDoc)
		if err := fn.AddKernel(binaryKernel(b, b, kleeneExec(op), exec.NullComputedPrealloc)); err != nil {
			panic(err)
		}
		addScalar(reg, parent, fn)
	}
	// ---- array_filter / array_take for the primitive types (selection.go:593-650): vector kernels, the kernel
	// allocates its own output (NullComputedNoPrealloc + MemNoPrealloc are the VectorKernel defaults, kernel.go:717-727).
	// The `filter` / `take` meta functions of the parent resolve "array_filter" / "array_take" through the registry
	// of the exec context, i.e. through this child.  Other value types keep the parent's kernels (see vectorDelegating).
	filterFn := compute.NewVectorFunction("array_filter", compute.Binary(), compute.EmptyFuncDoc)
	takeFn := compute.NewVectorFunction("array_take", compute.Binary(), compute.EmptyFuncDoc)
	for _, ty := range append(append([]arrow.DataType{}, numericTypes...), b) {
		fk := exec.NewVectorKernel([]exec.InputType{exec.NewExactInput(ty), exec.NewExactInput(b)}, kernels.OutputFirstType, filterExec,
			exec.OptionsInit[kernels.FilterState])
		if err := filterFn.AddKernel(fk); err != nil {
			panic(err)
		}
		tk := exec.NewVectorKernel([]exec.InputType{exec.NewExactInput(ty), exec.NewMatchedInput(exec.Integer())}, kernels.OutputFirstType, takeExec,
			exec.OptionsInit[kernels.TakeState])
		tk.CanExecuteChunkWise = false
		if err := takeFn.AddKernel(tk); err != nil {
			panic(err)
		}
	}
	addVector(reg, parent, filterFn)
	addVector(reg, parent, takeFn)
	registerLookupSort(reg, parent) // is_in, unique, dictionary_encode, sort_indices (lookup_sort.go)
	return reg
}

// vectorDelegating: same idea as delegating, for VectorFunctions.
type vectorDelegating struct {
	*compute.VectorFunction
	parent compute.Function
}

func (d *vectorDelegating) Execute(ctx context.Context, opts compute.FunctionOptions, args ...compute.Datum) (compute.Datum, error) {
	types := make([]arrow.DataType, len(args))
	for i, a := range args {
		types[i] = a.(compute.ArrayLikeDatum).Type()
	}
	if _, err := d.VectorFunction.DispatchExact(types...); err == nil {
		if opts == nil && d.parent != nil {
			opts = d.parent.DefaultOptions() // VectorFunction.defaultOpts is unexported (selection.go:618,636)
		}
		return d.VectorFunction.Execute(ctx, opts, args...)
	}
	if d.parent != nil {
		return d.parent.Execute(ctx, opts, args...)
	}
	return d.VectorFunction.Execute(ctx, opts, args...)
}

func (d *vectorDelegating) DefaultOptions() compute.FunctionOptions {
	if d.parent != nil {
		return d.parent.DefaultOptions()
	}
	return nil
}

func addVector(reg, parent compute.FunctionRegistry, fn *compute.VectorFunction) {
	p, _ := parent.GetFunction(fn.Name())
	reg.AddFunction(&vectorDelegating{VectorFunction: fn, parent: p}, true)
}
