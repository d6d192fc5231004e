// bamrec.cuh -- what the two readers of raw BAM records share (bamin.cu: the pileup's way in; bamdup.cu: duplicate marking
// of a file): little-endian loads, the name hash and the pairing of the two primary records of a name.
#pragma once
#include "pipeline.cuh"

__device__ __forceinline__ uint32_t qm_ld_u32(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
__device__ __forceinline__ uint32_t qm_ld_u16(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8; }

// FNV-1a over the read name of record r (without its NUL), cut to hash_bits bits (1..64; the tests force collisions with few bits)
__device__ __forceinline__ uint64_t qm_bam_name_hash(const uint8_t *r, int hash_bits)
{
    const int l_name = r[12];
    uint64_t h = 1469598103934665603ull;
    for (int i = 0; i + 1 < l_name; ++i) { h ^= r[36 + i]; h *= 1099511628211ull; }
    return hash_bits >= 64 ? h : h & ((1ull << hash_bits) - 1);
}

// a record that takes part in pairing: the first or the last segment, neither secondary (0x100) nor supplementary (0x800)
__device__ __forceinline__ bool qm_bam_pairing_primary(uint32_t flag)
{
    const uint32_t m = flag & 0xc0;
    return (m == 0x40 || m == 0x80) && !(flag & 0x900);
}

// bamin.cu: keys[k] = name hash, perm[k] = record index, sorted by hash (qm_sort_pairs); flags[f] = SAM flag of record f.
// partner[f] = the record f pairs with, -1 = none: f and g pair iff they are the only two pairing primaries of their name (names
// compared byte for byte) and one is the first, the other the last segment.
cudaError_t qm_bam_pair_launch(const uint8_t *d_bytes, const int64_t *d_rec_off, const uint16_t *d_flags, const uint64_t *d_keys,
                               const uint32_t *d_perm, int64_t n, int32_t *d_partner, cudaStream_t st);
