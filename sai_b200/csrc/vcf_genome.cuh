// Genome ingest (vcf_device.cu, driven by the engine's sai_engine_vcf_genome_* session): one pass over
// a multi-chromosome VCF keeps the records of every chromosome of a table.
#pragma once
#include "common.cuh"

namespace sai {

constexpr int kChromHashSlots = 2 * SAI_VCF_MAX_CHROMS;  // open addressing, load factor <= 1/2

// FNV-1a over the name's bytes (host: table build, device: CHROM lookup)
__host__ __device__ inline uint32_t chrom_hash(const char* p, int n) {
  uint32_t h = 2166136261u;
  for (int i = 0; i < n; ++i) h = (h ^ (uint8_t)p[i]) * 16777619u;
  return h;
}

struct VcfGenomeQuery {
  sai_vcf_query q;          // layout, sample columns, every chromosome's ancestral entries concatenated;
                            // chrom / start / end are not used
  const int64_t* anc_off;   // DEVICE [n_chrom + 1]: chromosome c's entries are anc_off[c] .. anc_off[c + 1]
  const char* names;        // DEVICE, the names back to back
  const int32_t* name_off;  // DEVICE [n_chrom + 1]
  const uint32_t* hash;     // DEVICE [2 * kChromHashSlots]: (hash, chromosome + 1) per slot, 0 = empty
  int32_t n_chrom;
};

// device-side running state of one genome parse (vcf_genome_state_init before the first slice)
struct VcfGenomeState {
  int64_t lines;          // lines of the slices parsed so far (file order of the span keys)
  int32_t last_chrom;     // chromosome of the last kept site, -1 before the first
  int32_t noncontiguous;  // 1: a chromosome's kept sites resumed after another chromosome's
};

struct VcfChromDev {
  unsigned long long first_key, last_key;  // (line << 32) | POS of the first / last record in file order
  int64_t n_records;                       // records of the chromosome, before the ancestral-allele filter
  int64_t first_site, n_sites;             // kept sites [first_site, first_site + n_sites); -1 / 0: none
};

// Negative-value table of an ingest session (DD, see N4 of sai_b200.h): the genotype pass keeps the raw
// value of every missing call.  Slices append their entries to `site/ind/val` in any order (one atomic
// per (record, population) with missing calls); each entry also gets its (chromosome, population) key
// and its index among that key's entries in (site, individual) order, which the slices derive from a
// scan of their per-(population, record) counts plus `count` (the key's entries of the slices before:
// slices run in stream order).  vcf_neg_order then places the entries key-major.
struct VcfNegDev {
  unsigned long long n;           // entries so far: the true count, also past cap (nothing is written there)
  unsigned long long slice_base;  // n when the current slice's genotype pass started
};
struct VcfNegSession {
  VcfNegDev* state;            // DEVICE
  unsigned long long* count;   // DEVICE [n_chrom][n_pops] entries so far per key
  int32_t *site, *ind, *val;   // DEVICE [cap] entries in append order (site: chromosome-local)
  int32_t *key, *idx;          // DEVICE [cap] chromosome * n_pops + population, index inside the key
  int64_t cap;
};

// The hash table of n names (name_off[n] bytes at `names`) into table[2 * kChromHashSlots];
// SAI_E_ARG for more than SAI_VCF_MAX_CHROMS names, an empty or a repeated name.
int vcf_chrom_table(const char* names, const int32_t* name_off, int32_t n, uint32_t* table);
int vcf_genome_state_init(VcfGenomeState* d_gs, VcfChromDev* d_chroms, int32_t n_chrom, cudaStream_t stream);
uint64_t vcf_genome_scratch_bytes(const VcfGenomeQuery& g, int64_t len);
// extra slice scratch of a session that keeps the negative-value table
uint64_t vcf_neg_scratch_bytes(const sai_vcf_query& q, int64_t len);
// sai_vcf_tiles_device for a chromosome table: kept sites numbered in file order, each chromosome's
// first site on a tile boundary, the sites between a chromosome's last site and that boundary coded
// all-missing.  d_state->n_sites is the end of the last chromosome's sites.  neg != NULL: the slice's
// negative-value entries are appended to it (scratch_bytes then includes vcf_neg_scratch_bytes).
int vcf_tiles_genome(const VcfGenomeQuery& g, const char* d_text, int64_t len, void* d_scratch, uint64_t scratch_bytes,
                     void* d_tiles, int32_t* d_pos, int64_t site_cap, sai_vcf_state* d_state, VcfGenomeState* d_gs,
                     VcfChromDev* d_chroms, const VcfNegSession* neg, cudaStream_t stream);
// sai_vcf_tiles_device with the negative-value table (neg != NULL) or without
int vcf_tiles_single(const sai_vcf_query& q, const char* d_text, int64_t len, void* d_scratch, uint64_t scratch_bytes,
                     void* d_tiles, int32_t* d_pos, int64_t site_cap, sai_vcf_state* d_state, const VcfNegSession* neg,
                     cudaStream_t stream);
// the n appended entries of `neg` -> out_site/ind/val, key k's entries from key_off[k] on (DEVICE)
int vcf_neg_order(const VcfNegSession& neg, int64_t n, const int64_t* d_key_off, int32_t* out_site, int32_t* out_ind,
                  int32_t* out_val, cudaStream_t stream);

}  // namespace sai
