package arrowgpu_test

import (
	"strings"
	"testing"

	"github.com/apache/arrow-go/v18/arrow"
	"github.com/apache/arrow-go/v18/arrow/array"
	"github.com/apache/arrow-go/v18/arrow/compute"
	"github.com/apache/arrow-go/v18/arrow/memory"
)

// vector_hash_test.go TestDictionaryEncode / TestDictionaryEncodeChunked on the GPU registry
func TestDictionaryEncodeOnDevice(t *testing.T) {
	mem := memory.NewCheckedAllocator(memory.DefaultAllocator)
	defer mem.AssertSize(t, 0)
	ctx := compute.WithAllocator(gpuCtx(), mem)

	vals, _, _ := array.FromJSON(mem, arrow.PrimitiveTypes.Int64, strings.NewReader(`[1, 2, 1, 3, 2]`))
	defer vals.Release()
	res, err := compute.CallFunction(ctx, "dictionary_encode", nil, compute.NewDatum(vals))
	if err != nil {
		t.Fatal(err)
	}
	defer res.Release()
	got := res.(compute.ArrayLikeDatum).Chunks()
	defer func() {
		for _, c := range got {
			c.Release()
		}
	}()
	wantIdx, _, _ := array.FromJSON(mem, arrow.PrimitiveTypes.Int32, strings.NewReader(`[0, 1, 0, 2, 1]`))
	defer wantIdx.Release()
	wantDict, _, _ := array.FromJSON(mem, arrow.PrimitiveTypes.Int64, strings.NewReader(`[1, 2, 3]`))
	defer wantDict.Release()
	d := got[0].(*array.Dictionary)
	if !array.Equal(d.Indices(), wantIdx) || !array.Equal(d.Dictionary(), wantDict) {
		t.Fatalf("dictionary_encode: got %v / %v", d.Indices(), d.Dictionary())
	}

	c1, _, _ := array.FromJSON(mem, arrow.PrimitiveTypes.Int32, strings.NewReader(`[1, 2, 1]`))
	c2, _, _ := array.FromJSON(mem, arrow.PrimitiveTypes.Int32, strings.NewReader(`[2, 3, null]`))
	chunked := arrow.NewChunked(arrow.PrimitiveTypes.Int32, []arrow.Array{c1, c2})
	c1.Release()
	c2.Release()
	defer chunked.Release()
	cres, err := compute.CallFunction(ctx, "dictionary_encode", nil, compute.NewDatum(chunked))
	if err != nil {
		t.Fatal(err)
	}
	defer cres.Release()
	chunks := cres.(*compute.ChunkedDatum).Value.Chunks()
	want := []string{`[0, 1, 0]`, `[1, 2, null]`}
	for i, c := range chunks {
		w, _, _ := array.FromJSON(mem, arrow.PrimitiveTypes.Int32, strings.NewReader(want[i]))
		if !array.Equal(c.(*array.Dictionary).Indices(), w) {
			t.Fatalf("chunk %d: got %v want %v", i, c.(*array.Dictionary).Indices(), w)
		}
		w.Release()
	}
}
