// TEST INFRASTRUCTURE ONLY. extern "C" hook over the stand-in CKMCFile (oracle/shim/kmc_file.h), the KMC reader
// the reference's main.cpp is compiled against in oracle/_ref.  It needs nothing outside this repository, so
// oracle/libkmc_shim.so is always built; tests/test_kmc_format_cpu.py checks it against the other two KMC readers.
#include <cstring>
#include <string>
#include <vector>

#include "kmc_file.h"

extern "C" {

// ---- KMC listing as call_main drives it (main.cpp:444-449, 482-490), through the stand-in CKMCFile -------------
// Writes "KMER\tCOUNT\n" lines; returns the text length (negative: buffer too small), -1 if the database cannot
// be opened.  info[0..7] = kmer_length, mode, counter_size, lut_prefix_length, signature_len, min_count, max_count,
// total_kmers as CKMCFile::Info reports them.
long shim_kmc_list(const char *prefix, uint64_t *info, char *out, long out_cap) {
  CKMCFile db;
  if (!db.OpenForListing(prefix)) return -1;
  uint32 klen = 0, mode = 0, csz = 0, lpl = 0, sl = 0, minc = 0;
  uint64 maxc = 0, total = 0;
  db.Info(klen, mode, csz, lpl, sl, minc, maxc, total);
  if (info) {
    info[0] = klen, info[1] = mode, info[2] = csz, info[3] = lpl, info[4] = sl, info[5] = minc, info[6] = maxc,
    info[7] = total;
  }
  CKmerAPI kmer_obj(klen);
  std::string res;
  uint32 counter;
  std::vector<char> context(klen + 1);
  while (db.ReadNextKmer(kmer_obj, counter)) {
    kmer_obj.to_string(context.data());
    res.append(context.data(), klen);
    res += '\t';
    res += std::to_string(counter);
    res += '\n';
  }
  if ((long)res.size() + 1 > out_cap) return -(long)res.size() - 2;
  memcpy(out, res.c_str(), res.size() + 1);
  return (long)res.size();
}

}  // extern "C"
