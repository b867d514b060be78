// blu_sort.h -- the stable radix sort of blu_sort.cu and the ordering of result records by query id built on it.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/blu_consensus.h"

namespace blu {

// Stable sort of (keys, vals) by the low `bits` bits of the keys (LSD, 8-bit digits).  The four arrays hold n elements each;
// the sorted pairs end in (keys, vals) (*in_alt == false) or in (keys_alt, vals_alt) (*in_alt == true).  `scratch` holds
// radix_sort_scratch_bytes(n) bytes of device memory.  Synchronises `s` once to skip digits that every key shares.
size_t radix_sort_scratch_bytes(uint32_t n);
cudaError_t radix_sort_pairs_u32(uint32_t* keys, uint32_t* keys_alt, uint32_t* vals, uint32_t* vals_alt, uint32_t n, int bits, void* scratch,
                                 cudaStream_t s, bool* in_alt);

// Device bytes sort_ids_device() allocates for n ids.
uint64_t sort_ids_device_bytes(uint64_t n);
// perm[i] = the index of the id that goes to position i when ids are ordered bytewise (unsigned, a prefix first), equal ids in
// their order of index.  Id i is base[off[i] .. off[i] + len[i]) in device memory.  0: done; 1: the scratch does not fit the
// device; < 0: a CUDA error (cudaError_t negated).
int sort_ids_device(const uint8_t* base, const uint64_t* off, const uint32_t* len, uint32_t n, uint32_t* perm, cudaStream_t s);
// off[i] / len[i] = the query id reference of rec[i]
cudaError_t launch_record_ids(const blu_record* rec, uint32_t n, uint64_t* off, uint32_t* len, cudaStream_t s);
// out[i] = in[perm[i]]
cudaError_t launch_gather_records(const blu_record* in, const uint32_t* perm, uint32_t n, blu_record* out, cudaStream_t s);

}  // namespace blu
