// Host build of the counter-based dropout definition in csrc/gemm_epilogue.cuh (drop_key_mixed / drop_epoch_seed /
// drop_thr16 / drop_inv_keep / drop_keep), for tests/test_host_dropout.py: the numpy reference (tests/dropout_ref.py)
// is compared with the very code the kernels compile.
//
//   dropout_host <seed> <epoch> <p> <G>   (decimal, p as a float)
//   stdin : n little-endian uint64 element indices
//   stdout: uint32 thr16, float32 inv_keep, then n bytes (1 = kept)
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "gemm_epilogue.cuh"

int main(int argc, char** argv) {
  if (argc != 5) {
    fprintf(stderr, "usage: %s seed epoch p G < indices.u64 > keep.u8\n", argv[0]);
    return 2;
  }
  const unsigned long long seed = strtoull(argv[1], nullptr, 10), epoch = strtoull(argv[2], nullptr, 10);
  const float p = strtof(argv[3], nullptr);
  const int G = atoi(argv[4]);
  if (G != 8 && G != 16) {
    fprintf(stderr, "G must be 8 or 16\n");
    return 2;
  }
  const DropKey k = drop_key_mixed(drop_epoch_seed(seed, epoch), p);
  fwrite(&k.thr16, 4, 1, stdout);
  fwrite(&k.inv_keep, 4, 1, stdout);
  std::vector<unsigned long long> idx(1 << 16);
  std::vector<unsigned char> keep(idx.size());
  size_t n;
  while ((n = fread(idx.data(), 8, idx.size(), stdin)) > 0) {
    for (size_t i = 0; i < n; ++i) keep[i] = (G == 8 ? drop_keep<8>(k, idx[i]) : drop_keep<16>(k, idx[i])) ? 1 : 0;
    fwrite(keep.data(), 1, n, stdout);
  }
  return 0;
}
