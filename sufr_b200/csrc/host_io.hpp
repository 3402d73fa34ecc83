// Host-side pieces of the create path: SeedMask, the `.sufr` writer and FASTA/FASTQ ingest.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/sufr_b200.h"

namespace sufr {

// libsufr/src/types.rs:36-200
struct SeedMaskInfo {
    std::string mask;
    std::vector<uint8_t> bytes;
    std::vector<uint64_t> positions;
    uint64_t weight = 0;
};
bool parse_seed_mask(const char* mask, SeedMaskInfo& out);
uint64_t lcp_full_offset(uint64_t lcp, const SeedMaskInfo& m);  // util.rs:19-37

// sufr_builder.rs:817-918
void write_sufr_file(const SufrB200Args& args, const SufrB200Result& r);

// The parts of a version-6 `.sufr` file around the three big sections (sufr_builder.rs:826-867, :909).
struct SufrFrame {
    std::vector<uint8_t> head;  // everything before the text
    std::vector<uint8_t> tail;  // bincode Vec<String> of the sequence names
    uint64_t text_pos = 0, sa_pos = 0, lcp_pos = 0, names_pos = 0;
};
SufrFrame make_sufr_frame(const SufrB200Args& args, uint32_t index_bits, uint64_t text_len, uint64_t total_suffixes);
void pwrite_all(int fd, const void* buf, size_t len, uint64_t off, const std::string& path);

// The header, sequence starts, seed mask and names tail of a version-6 `.sufr` file (read side of the layout above,
// sufr_file.rs:145-275), validated so that every section offset and every sequence start can be trusted: a file that
// fails a check is refused with SUFR_B200_ERR_IO ("{path}: invalid .sufr file: ..."), a version other than 6 with
// SUFR_B200_ERR_UNSUPPORTED.  The three big sections are not read.
struct SufrFileInfo {
    uint32_t version = 0, index_bits = 0;
    bool is_dna = false, allow_ambiguity = false, ignore_softmask = false;
    uint64_t text_len = 0, num_suffixes = 0, max_query_len = 0;
    uint64_t text_pos = 0, sa_pos = 0, lcp_pos = 0, file_bytes = 0;
    std::string seed_mask;  // "" = none
    std::vector<uint64_t> sequence_starts;
    std::vector<std::string> sequence_names;
};
void read_sufr_info(const std::string& path, SufrFileInfo& out);
void pread_all(int fd, void* buf, size_t len, uint64_t off, const std::string& path);

// The output file of a build, written by many threads (and, sharded, by several ranks) at known offsets.  Concurrent
// pwrite()s to ONE file serialise on the inode lock (3.5 GB/s on a RAM disk, whatever the thread count), so the file is
// sized up front and mapped: the writers copy into the mapping and fault its pages in parallel.  Falls back to pwrite
// where the file cannot be mapped.
class OutputFile {
   public:
    OutputFile(const std::string& path, uint64_t final_size, bool truncate_existing);
    ~OutputFile();
    OutputFile(const OutputFile&) = delete;
    OutputFile& operator=(const OutputFile&) = delete;
    void write(uint64_t off, const void* buf, size_t len);            // thread-safe for disjoint ranges
    void write_parallel(uint64_t off, const void* buf, size_t len);   // a large section, copied by several threads
    void close();                                                     // reports errors; the destructor does not
    bool mapped() const { return map_ != nullptr; }

   private:
    std::string path_;
    int fd_ = -1;
    uint8_t* map_ = nullptr;
    uint64_t size_ = 0;
};

// util.rs:51-89
void read_sequence_file(const char* path, uint8_t delim, SufrB200Sequences* out);
void free_sequences(SufrB200Sequences* s);

}  // namespace sufr
