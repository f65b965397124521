// psb_db.h -- the resident database object shared by engine.cu (construction, scans) and db_io.cu
// (FASTA reader, on-disk packed format).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <mutex>
#include <vector>

struct psb_db {
    int device = 0;
    cudaStream_t stream = nullptr;  // stream the buffers were allocated on (stream-ordered pool)
    int64_t n = 0, residues = 0, words = 0;
    int bits = 5;                   // 2, 3 or 5 bits per residue (16, 10 or 6 residues per 32-bit word)
    int msize = 0;
    int maxlen = 0;                 // longest subject
    int nlong = 0;                  // subjects longer than 65535 (sorted first)
    std::vector<int> top_len;       // lengths of the (up to 4096) longest subjects, descending
    std::vector<int> host_len;      // caller-order lengths (psb_db_create / psb_db_load only; explicit-width saturation flags)
    uint8_t mapper[256];
    unsigned *d_words = nullptr;
    long long *d_word_off = nullptr;  // n+1, sorted order (length descending, stable)
    int *d_perm = nullptr;            // sorted position -> caller's subject id
    int *d_len = nullptr;             // sorted order
    long long *d_res_off = nullptr;   // n+1 prefix sum of d_len: boundary lines of the strip-wise scan (built on first use)
    int *d_inv_perm = nullptr;        // caller's subject id -> sorted position (built on first use by psb_db_align / psb_db_subject)
    std::mutex mu;
};

namespace psb {
// bits per residue of a packed database for an alphabet of `size` letters (pad / wildcard codes are < size)
inline int db_bits_for(int size) { return size <= 4 ? 2 : (size <= 8 ? 3 : 5); }
inline int db_residues_per_word(int bits) { return bits == 2 ? 16 : (bits == 3 ? 10 : 6); }
// engine.cu: binds the calling thread's context (device, stream); PSB_OK or an error code
int db_io_ensure_ctx(int *device, cudaStream_t *stream);
}  // namespace psb
