// Shared pieces of the ordered (deterministic) reductions, see ordered.cu.
#pragma once
#include "common.cuh"

namespace neko {

constexpr int ORD_ROWS = 64;          // rows per fixed block of the column sums

// Destination of an ordered column reduction: columns [off[i], off[i+1]) of the workspace rows go to p[i][0 ..].
struct OrdDst {
  float* p[6];
  int off[7];
  int n;
};

// dst(c) (+)= sum over b = 0 .. n_blocks-1 of ws[b * ld + c], c < ncols, in a fixed order that depends on n_blocks only.
int ordered_colreduce(const float* ws, long long ld, int n_blocks, int ncols, const OrdDst& dst, int accumulate, cudaStream_t st);
// Grid of a launch over `units` fixed work units: all of them, or NEKO_ORDERED_CTAS when that is smaller (the result does not
// depend on it; tests use it to show so).
int ordered_grid(long long units);

// Sorted scatter-add into up to three tables: key k in [off[i], off[i+1]) adds into row k - off[i] of p[i] ([rows, d] fp32);
// keys >= off[3] are skipped.
struct SegDst {
  float* p[3];
  int off[4];
};
// Workspace of a stable radix sort of n (key, value) pairs with keys below 2^end_bit: input and output arrays, then the sort's
// own scratch.  base == nullptr computes the sizes only (s.total).
struct SortWs {
  unsigned* kin;
  int* vin;
  unsigned* kout;
  int* vout;
  void* temp;
  size_t temp_bytes;
  size_t total;
};
int key_bits(unsigned max_key);
int sort_ws_layout(long long n, int end_bit, void* base, SortWs& s);
// Sorts s.kin / s.vin (values = source rows of src [*, d]) and adds, for every key, the sum of its source rows taken in
// ascending order to the key's table row.
int sort_and_segsum(SortWs& s, long long n, int end_bit, const float* src, int d, const SegDst& dst, cudaStream_t st);

}  // namespace neko
