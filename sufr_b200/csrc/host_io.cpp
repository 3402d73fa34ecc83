#include "host_io.hpp"

#include <dlfcn.h>
#include <fcntl.h>
#include <zlib.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

namespace sufr {

// ------------------------------------------------------------------ SeedMask (types.rs:80-200)
bool parse_seed_mask(const char* mask, SeedMaskInfo& out) {
    // valid iff it matches ^1+0[01]*1$ (types.rs:163-166): only 0/1, starts and ends with 1, has a 0
    size_t len = strlen(mask);
    if (len < 3 || mask[0] != '1' || mask[len - 1] != '1') return false;
    bool zero = false;
    for (size_t i = 0; i < len; i++) {
        if (mask[i] == '0') zero = true;
        else if (mask[i] != '1') return false;
    }
    if (!zero) return false;
    out.mask = mask;
    out.bytes.clear();
    out.positions.clear();
    for (size_t i = 0; i < len; i++) {
        out.bytes.push_back(mask[i] == '1' ? 1 : 0);
        if (mask[i] == '1') out.positions.push_back(i);
    }
    out.weight = out.positions.size();
    return true;
}

uint64_t lcp_full_offset(uint64_t lcp, const SeedMaskInfo& m) {
    if (lcp == 0 || lcp > m.bytes.size()) return lcp;
    uint64_t offset = m.positions[lcp - 1];
    uint64_t next_offset = lcp < m.positions.size() ? m.positions[lcp] : 0;
    if (next_offset > offset && next_offset - offset > 1) return next_offset;
    return offset + 1;
}

// ------------------------------------------------------------------ `.sufr` writer
static void put_u64(std::vector<uint8_t>& out, uint64_t v) {  // util.rs:138-151
    for (int i = 0; i < 8; i++) out.push_back((uint8_t)(v >> (8 * i)));
}

void pwrite_all(int fd, const void* buf, size_t len, uint64_t off, const std::string& path) {
    const char* p = (const char*)buf;
    while (len) {
        size_t chunk = len > (1u << 30) ? (1u << 30) : len;
        ssize_t w = pwrite(fd, p, chunk, (off_t)off);
        if (w < 0) {
            if (errno == EINTR) continue;
            throw Error(SUFR_B200_ERR_IO, path + ": " + strerror(errno));
        }
        p += w;
        off += (uint64_t)w;
        len -= (size_t)w;
    }
}

SufrFrame make_sufr_frame(const SufrB200Args& args, uint32_t index_bits, uint64_t text_len, uint64_t total_suffixes) {
    SufrFrame f;
    const size_t w = index_bits / 8;
    if (args.num_sequences && !args.sequence_starts)
        throw Error(SUFR_B200_ERR_ARGUMENT, "sequence_starts is NULL but num_sequences > 0");
    if (args.num_sequences && args.sequence_names)
        for (uint64_t i = 0; i < args.num_sequences; i++)
            if (!args.sequence_names[i]) throw Error(SUFR_B200_ERR_ARGUMENT, "sequence_names holds a NULL entry");
    SeedMaskInfo mask;
    const bool has_mask = args.seed_mask && parse_seed_mask(args.seed_mask, mask);

    // header (sufr_builder.rs:826-867); all integers little-endian
    std::vector<uint8_t>& head = f.head;
    head.push_back(6);  // OUTFILE_VERSION, types.rs:16
    head.push_back(args.is_dna ? 1 : 0);
    head.push_back(args.allow_ambiguity ? 1 : 0);
    head.push_back(args.ignore_softmask ? 1 : 0);
    put_u64(head, text_len);
    const size_t locs_pos = head.size();
    put_u64(head, 0);
    put_u64(head, 0);
    put_u64(head, 0);
    put_u64(head, total_suffixes);
    put_u64(head, has_mask ? 0 : (args.has_max_query_len ? args.max_query_len : 0));
    put_u64(head, args.num_sequences);
    for (uint64_t i = 0; i < args.num_sequences; i++) {
        uint64_t v = args.sequence_starts[i];
        for (size_t k = 0; k < w; k++) head.push_back((uint8_t)(v >> (8 * k)));
    }
    if (has_mask) {
        put_u64(head, mask.bytes.size());
        head.insert(head.end(), mask.bytes.begin(), mask.bytes.end());
    } else {
        put_u64(head, 0);
    }
    f.text_pos = head.size();
    f.sa_pos = f.text_pos + text_len;
    f.lcp_pos = f.sa_pos + total_suffixes * w;
    f.names_pos = f.lcp_pos + total_suffixes * w;
    {
        std::vector<uint8_t> locs;
        put_u64(locs, f.text_pos);
        put_u64(locs, f.sa_pos);
        put_u64(locs, f.lcp_pos);
        memcpy(head.data() + locs_pos, locs.data(), locs.size());
    }
    // bincode 1.3 Vec<String>: u64 count, then per string u64 length + bytes (sufr_builder.rs:909)
    put_u64(f.tail, args.num_sequences);
    for (uint64_t i = 0; i < args.num_sequences; i++) {
        const char* nm = args.sequence_names ? args.sequence_names[i] : "";
        size_t len = strlen(nm);
        put_u64(f.tail, len);
        f.tail.insert(f.tail.end(), nm, nm + len);
    }
    return f;
}

OutputFile::OutputFile(const std::string& path, uint64_t final_size, bool truncate_existing) : path_(path), size_(final_size) {
    fd_ = open(path.c_str(), O_RDWR | O_CREAT | (truncate_existing ? O_TRUNC : 0), 0644);
    if (fd_ < 0) throw Error(SUFR_B200_ERR_IO, path + ": " + strerror(errno));  // sufr_builder.rs:820
    // every writer (rank) sets the same final size: idempotent, and no rank has to wait for another one
    if (ftruncate(fd_, (off_t)final_size) != 0) {
        const std::string msg = path + ": " + strerror(errno);
        ::close(fd_);
        fd_ = -1;
        throw Error(SUFR_B200_ERR_IO, msg);
    }
    if (final_size && !getenv("SUFR_B200_DEBUG_NO_MMAP")) {
        void* m = mmap(nullptr, final_size, PROT_READ | PROT_WRITE, MAP_SHARED, fd_, 0);
        if (m != MAP_FAILED) map_ = (uint8_t*)m;
    }
}

OutputFile::~OutputFile() {
    if (map_) munmap(map_, size_);
    if (fd_ >= 0) ::close(fd_);
}

void OutputFile::close() {
    if (map_) {
        if (munmap(map_, size_) != 0) { map_ = nullptr; throw Error(SUFR_B200_ERR_IO, path_ + ": " + strerror(errno)); }
        map_ = nullptr;
    }
    if (fd_ >= 0) {
        const int rc = ::close(fd_);
        fd_ = -1;
        if (rc != 0) throw Error(SUFR_B200_ERR_IO, path_ + ": " + strerror(errno));
    }
}

void OutputFile::write(uint64_t off, const void* buf, size_t len) {
    if (len == 0) return;
    if (off + len > size_) throw Error(SUFR_B200_ERR_INTERNAL, path_ + ": write beyond the planned file size");
    if (map_) memcpy(map_ + off, buf, len);
    else pwrite_all(fd_, buf, len, off, path_);
}

// A section of tens of GB copied by several threads (page-cache copies are CPU bound: page allocation + memcpy).
void OutputFile::write_parallel(uint64_t off, const void* buf, size_t len) {
    size_t piece = 64u << 20;
    if (const char* dbg = getenv("SUFR_B200_DEBUG_WRITE_PIECE")) piece = std::max<size_t>(1, strtoull(dbg, nullptr, 10));
    size_t T = std::thread::hardware_concurrency();
    T = std::max<size_t>(1, std::min<size_t>(std::min<size_t>(T, 24), len / piece));
    if (T <= 1) { write(off, buf, len); return; }
    std::vector<std::thread> pool;
    std::vector<std::exception_ptr> err(T);
    for (size_t t = 0; t < T; t++)
        pool.emplace_back([&, t]() {
            try {
                const size_t lo = len * t / T, hi = len * (t + 1) / T;
                write(off + lo, (const char*)buf + lo, hi - lo);
            } catch (...) { err[t] = std::current_exception(); }
        });
    for (auto& th : pool) th.join();
    for (auto& e : err) if (e) std::rethrow_exception(e);
}

void write_sufr_file(const SufrB200Args& args, const SufrB200Result& r) {
    const std::string path = args.path ? args.path : "out.sufr";  // sufr_builder.rs:215
    const size_t w = r.index_bits / 8;
    const SufrFrame f = make_sufr_frame(args, r.index_bits, r.text_len, r.total_suffixes);
    const bool sharded = args.world_size > 1;
    const bool leader = !sharded || args.rank == 0;
    OutputFile out(path, f.names_pos + f.tail.size(), !sharded);
    if (leader) {
        out.write(0, f.head.data(), f.head.size());
        out.write_parallel(f.text_pos, r.text, r.text_len);
        out.write(f.names_pos, f.tail.data(), f.tail.size());
    }
    out.write_parallel(f.sa_pos + r.shard_offset * w, r.sa, r.num_suffixes * w);
    out.write_parallel(f.lcp_pos + r.shard_offset * w, r.lcp, r.num_suffixes * w);
    out.close();
}

// ------------------------------------------------------------------ `.sufr` reader (header, starts, mask, names)
void pread_all(int fd, void* buf, size_t len, uint64_t off, const std::string& path) {
    char* p = (char*)buf;
    while (len) {
        const ssize_t got = pread(fd, p, std::min<size_t>(len, 1u << 30), (off_t)off);
        if (got < 0 && errno == EINTR) continue;
        if (got < 0) throw Error(SUFR_B200_ERR_IO, path + ": " + strerror(errno));
        if (got == 0) throw Error(SUFR_B200_ERR_IO, path + ": invalid .sufr file: unexpected end of file");
        p += got;
        off += (uint64_t)got;
        len -= (size_t)got;
    }
}

static uint64_t get_u64(const uint8_t* p) {
    uint64_t v = 0;
    for (int i = 7; i >= 0; i--) v = (v << 8) | p[i];
    return v;
}

void read_sufr_info(const std::string& path, SufrFileInfo& info) {
    info = SufrFileInfo();
    const int fd = open(path.c_str(), O_RDONLY);
    if (fd < 0) throw Error(SUFR_B200_ERR_IO, path + ": " + strerror(errno));
    struct FdCloser { int fd; ~FdCloser() { close(fd); } } closer{fd};
    auto bad = [&](const std::string& what) { return Error(SUFR_B200_ERR_IO, path + ": invalid .sufr file: " + what); };
    struct stat st;
    if (fstat(fd, &st) != 0) throw Error(SUFR_B200_ERR_IO, path + ": " + strerror(errno));
    if (!S_ISREG(st.st_mode)) throw bad("not a regular file");
    const uint64_t size = (uint64_t)st.st_size;
    info.file_bytes = size;
    if (size == 0) throw bad("empty file");
    uint8_t head[60];
    pread_all(fd, head, 1, 0, path);
    info.version = head[0];
    if (info.version != 6)
        throw Error(SUFR_B200_ERR_UNSUPPORTED,
                    path + ": unsupported .sufr version " + std::to_string(info.version) + " (only version 6 is read)");
    if (size < 60 + 8) throw bad("truncated header (" + std::to_string(size) + " bytes)");
    pread_all(fd, head, 60, 0, path);
    // sufr_builder.rs:826-867
    info.is_dna = head[1] != 0;
    info.allow_ambiguity = head[2] != 0;
    info.ignore_softmask = head[3] != 0;
    info.text_len = get_u64(head + 4);
    info.text_pos = get_u64(head + 12);
    info.sa_pos = get_u64(head + 20);
    info.lcp_pos = get_u64(head + 28);
    info.num_suffixes = get_u64(head + 36);
    info.max_query_len = get_u64(head + 44);
    const uint64_t nseq = get_u64(head + 52);
    const uint64_t n = info.text_len, s = info.num_suffixes;
    if (n > size || s > size) throw bad("text length / suffix count larger than the file");
    if (s > n) throw bad("num_suffixes " + std::to_string(s) + " exceeds the text length " + std::to_string(n));

    // element width: from the section sizes (--index-bits 64 writes u64 files of short texts); with no suffixes the
    // reference's rule (u32 iff text_len < u32::MAX, suffix_array.rs:460-470)
    uint64_t w;
    if (s > 0) {
        if (info.lcp_pos < info.sa_pos || (info.lcp_pos - info.sa_pos) % s != 0) throw bad("suffix array section size");
        w = (info.lcp_pos - info.sa_pos) / s;
        if (w != 4 && w != 8) throw bad("element width " + std::to_string(w) + " (must be 4 or 8 bytes)");
    } else {
        w = n < 0xFFFFFFFFull ? 4 : 8;
    }
    info.index_bits = (uint32_t)(w * 8);
    if (nseq > (size - 68) / w) throw bad("num_sequences " + std::to_string(nseq) + " does not fit the file");

    // sequence starts, then the seed mask (u64 length + one byte per position)
    std::vector<uint8_t> buf(nseq * w + 8);
    pread_all(fd, buf.data(), buf.size(), 60, path);
    info.sequence_starts.resize(nseq);
    for (uint64_t i = 0; i < nseq; i++) {
        uint64_t v = 0;
        for (int k = (int)w - 1; k >= 0; k--) v = (v << 8) | buf[i * w + k];
        info.sequence_starts[i] = v;
        if (v >= n) throw bad("sequence start " + std::to_string(v) + " is not below the text length");
        if (i > 0 && v <= info.sequence_starts[i - 1]) throw bad("sequence starts are not strictly increasing");
    }
    const uint64_t mask_off = 60 + nseq * w;
    const uint64_t mask_len = get_u64(buf.data() + nseq * w);
    if (mask_len > size - mask_off - 8) throw bad("seed mask length " + std::to_string(mask_len) + " does not fit the file");
    if (mask_len) {
        std::vector<uint8_t> mb(mask_len);
        pread_all(fd, mb.data(), mask_len, mask_off + 8, path);
        std::string mask(mask_len, '0');
        for (uint64_t i = 0; i < mask_len; i++) {
            if (mb[i] > 1) throw bad("seed mask byte " + std::to_string(mb[i]) + " (must be 0 or 1)");
            mask[i] = mb[i] ? '1' : '0';
        }
        SeedMaskInfo m;
        if (!parse_seed_mask(mask.c_str(), m)) throw bad("invalid seed mask '" + mask + "'");
        info.seed_mask = mask;
    }

    // the sections follow each other without gaps (sufr_builder.rs:841-867)
    if (info.text_pos != mask_off + 8 + mask_len)
        throw bad("text_pos " + std::to_string(info.text_pos) + " (expected " + std::to_string(mask_off + 8 + mask_len) + ")");
    if (info.sa_pos != info.text_pos + n)
        throw bad("sa_pos " + std::to_string(info.sa_pos) + " (expected " + std::to_string(info.text_pos + n) + ")");
    if (info.lcp_pos != info.sa_pos + s * w)
        throw bad("lcp_pos " + std::to_string(info.lcp_pos) + " (expected " + std::to_string(info.sa_pos + s * w) + ")");
    const uint64_t names_pos = info.lcp_pos + s * w;
    if (names_pos > size) throw bad("truncated (no sequence names after the LCP array)");

    // names: bincode Vec<String> up to exactly the end of the file (sufr_builder.rs:909), read through a small buffer
    // as they are parsed, so that a file with junk behind its names is refused without reading the junk
    struct TailReader {
        int fd;
        const std::string& path;
        uint64_t pos, end;
        std::vector<uint8_t> buf;
        size_t at = 0;
        bool take(void* dst, uint64_t len) {  // false: the file ends first
            if (len > end - pos + (buf.size() - at)) return false;
            uint8_t* d = (uint8_t*)dst;
            while (len) {
                if (at == buf.size()) {
                    buf.resize((size_t)std::min<uint64_t>(1u << 20, end - pos));
                    pread_all(fd, buf.data(), buf.size(), pos, path);
                    pos += buf.size();
                    at = 0;
                }
                const size_t k = (size_t)std::min<uint64_t>(len, buf.size() - at);
                memcpy(d, buf.data() + at, k);
                d += k;
                at += k;
                len -= k;
            }
            return true;
        }
        uint64_t left() const { return end - pos + (buf.size() - at); }
    } tail{fd, path, names_pos, size, {}};
    uint8_t word[8];
    if (!tail.take(word, 8)) throw bad("truncated (no sequence names after the LCP array)");
    const uint64_t count = get_u64(word);
    if (count != nseq)
        throw bad("the names tail holds " + std::to_string(count) + " names for " + std::to_string(nseq) + " sequences");
    info.sequence_names.reserve(nseq);
    for (uint64_t i = 0; i < nseq; i++) {
        if (!tail.take(word, 8)) throw bad("truncated sequence names");
        const uint64_t len = get_u64(word);
        if (len > tail.left()) throw bad("truncated sequence names");
        std::string name((size_t)len, '\0');
        tail.take(&name[0], len);
        info.sequence_names.push_back(std::move(name));
    }
    if (tail.left()) throw bad(std::to_string(tail.left()) + " unexpected bytes after the sequence names");
}

// ------------------------------------------------------------------ FASTA / FASTQ ingest (util.rs:51-89)
// The reference delegates parsing to needletail 0.6 (not vendored).  This follows its documented
// behaviour for plain-text input: FASTA records may span lines, FASTQ records are 4 lines, '\r' is
// stripped at line ends, the id is the header up to the first whitespace.
//
// Compressed input (needletail decompresses gz / bz2 / xz / zstd transparently): detected by magic bytes and inflated
// in memory -- gzip through zlib (multi-member files included), the other three through the system's runtime
// libraries (libbz2.so.1.0, liblzma.so.5, libzstd.so.1; loaded on demand, a clear error when one is missing).
//
// Both formats are parsed by all host cores: the file is read with parallel preads, cut into slices at record
// boundaries that can be recognised locally, and every slice is handled in two passes (count, then write at its
// final offset), so a 3 Gbp genome is ingested at memory speed instead of by one core.  FASTA slices start at any
// line start; a FASTQ slice starts at a line that begins with '@' and whose second successor begins with '+' (in a
// four-line record only the header satisfies both: a quality line that begins with '@' is followed by a header and
// then by a sequence line, which cannot begin with '+').
namespace {

struct FileData {
    char* p = nullptr;
    size_t n = 0;
    ~FileData() { free(p); }
};

int ingest_threads(size_t bytes) {
    size_t t = std::thread::hardware_concurrency();
    if (t == 0) t = 1;
    if (t > 32) t = 32;
    size_t by_size = bytes / (4u << 20) + 1;  // no point in a thread per few MB
    return (int)std::min(t, by_size);
}

template <typename F>
void parallel_for(int threads, F f) {
    if (threads <= 1) { f(0); return; }
    std::vector<std::thread> pool;
    std::vector<std::exception_ptr> err(threads);
    for (int t = 0; t < threads; t++)
        pool.emplace_back([&, t]() { try { f(t); } catch (...) { err[t] = std::current_exception(); } });
    for (auto& th : pool) th.join();
    for (auto& e : err) if (e) std::rethrow_exception(e);
}

// ---- decompression
struct Inflated {
    char* p = nullptr;
    size_t n = 0, cap = 0;
    void need(size_t extra) {
        if (n + extra <= cap) return;
        size_t c = std::max<size_t>(cap * 2, n + extra + (1u << 20));
        char* q = (char*)realloc(p, c);
        if (!q) { free(p); p = nullptr; throw Error(SUFR_B200_ERR_OUT_OF_MEMORY, "out of host memory while decompressing"); }
        p = q;
        cap = c;
    }
};

void inflate_gzip(const char* path, const char* src, size_t n, Inflated& out) {
    size_t pos = 0;
    while (pos < n) {  // one iteration per gzip member (bgzip and `cat a.gz b.gz` files have many)
        z_stream zs;
        memset(&zs, 0, sizeof(zs));
        if (inflateInit2(&zs, 16 + MAX_WBITS) != Z_OK) throw Error(SUFR_B200_ERR_INTERNAL, "zlib: inflateInit2 failed");
        int rc = Z_OK;
        while (rc != Z_STREAM_END) {
            out.need(4u << 20);
            zs.next_in = (Bytef*)(src + pos);
            zs.avail_in = (uInt)std::min<size_t>(n - pos, 1u << 30);
            zs.next_out = (Bytef*)(out.p + out.n);
            zs.avail_out = (uInt)std::min<size_t>(out.cap - out.n, 1u << 30);
            const uInt in0 = zs.avail_in, out0 = zs.avail_out;
            rc = inflate(&zs, Z_NO_FLUSH);
            pos += in0 - zs.avail_in;
            out.n += out0 - zs.avail_out;
            if (rc != Z_OK && rc != Z_STREAM_END && rc != Z_BUF_ERROR) {
                inflateEnd(&zs);
                throw Error(SUFR_B200_ERR_IO, std::string(path) + ": corrupt gzip data (" + (zs.msg ? zs.msg : "zlib error") + ")");
            }
            if (rc != Z_STREAM_END && pos >= n && in0 == zs.avail_in && out0 == zs.avail_out) {
                inflateEnd(&zs);
                throw Error(SUFR_B200_ERR_IO, std::string(path) + ": truncated gzip data");
            }
        }
        inflateEnd(&zs);
        while (pos < n && src[pos] == 0) pos++;  // zero padding between / behind members
    }
}

void* runtime_lib(const char* path, const char* const* names) {
    for (; *names; names++)
        if (void* h = dlopen(*names, RTLD_NOW | RTLD_GLOBAL)) return h;
    throw Error(SUFR_B200_ERR_UNSUPPORTED, std::string(path) + ": this input needs a decompression library that is not installed");
}
template <typename F>
F runtime_sym(void* lib, const char* name) {
    void* f = dlsym(lib, name);
    if (!f) throw Error(SUFR_B200_ERR_UNSUPPORTED, std::string("missing symbol ") + name);
    return reinterpret_cast<F>(f);
}

void inflate_zstd(const char* path, const char* src, size_t n, Inflated& out) {
    static const char* const names[] = {"libzstd.so.1", "libzstd.so", nullptr};
    void* lib = runtime_lib(path, names);
    auto content_size = runtime_sym<unsigned long long (*)(const void*, size_t)>(lib, "ZSTD_getFrameContentSize");
    auto frame_size = runtime_sym<size_t (*)(const void*, size_t)>(lib, "ZSTD_findFrameCompressedSize");
    auto decompress = runtime_sym<size_t (*)(void*, size_t, const void*, size_t)>(lib, "ZSTD_decompress");
    auto is_error = runtime_sym<unsigned (*)(size_t)>(lib, "ZSTD_isError");
    size_t pos = 0;
    while (pos < n) {  // one iteration per frame
        const size_t fs = frame_size(src + pos, n - pos);
        if (is_error(fs)) throw Error(SUFR_B200_ERR_IO, std::string(path) + ": corrupt zstd data");
        unsigned long long cs = content_size(src + pos, fs);
        size_t guess = cs < (1ull << 62) ? (size_t)cs : fs * 8 + (1u << 20);  // unknown size: grow until it fits
        for (;;) {
            out.need(guess);
            const size_t got = decompress(out.p + out.n, out.cap - out.n, src + pos, fs);
            if (!is_error(got)) { out.n += got; break; }
            if (cs < (1ull << 62) || guess > (1ull << 40)) throw Error(SUFR_B200_ERR_IO, std::string(path) + ": corrupt zstd data");
            guess *= 2;
        }
        pos += fs;
    }
}

void inflate_bzip2(const char* path, const char* src, size_t n, Inflated& out) {
    static const char* const names[] = {"libbz2.so.1.0", "libbz2.so.1", "libbz2.so", nullptr};
    void* lib = runtime_lib(path, names);
    // bz_stream of bzlib.h 1.0.x
    struct BzStream {
        char* next_in; unsigned avail_in, total_in_lo32, total_in_hi32;
        char* next_out; unsigned avail_out, total_out_lo32, total_out_hi32;
        void* state; void* (*bzalloc)(void*, int, int); void (*bzfree)(void*, void*); void* opaque;
    };
    auto init = runtime_sym<int (*)(BzStream*, int, int)>(lib, "BZ2_bzDecompressInit");
    auto step = runtime_sym<int (*)(BzStream*)>(lib, "BZ2_bzDecompress");
    auto end = runtime_sym<int (*)(BzStream*)>(lib, "BZ2_bzDecompressEnd");
    size_t pos = 0;
    while (pos < n) {  // one iteration per stream
        BzStream bz;
        memset(&bz, 0, sizeof(bz));
        if (init(&bz, 0, 0) != 0) throw Error(SUFR_B200_ERR_INTERNAL, "bzip2: init failed");
        int rc = 0;
        while (rc != 4 /* BZ_STREAM_END */) {
            out.need(4u << 20);
            bz.next_in = const_cast<char*>(src + pos);
            bz.avail_in = (unsigned)std::min<size_t>(n - pos, 1u << 30);
            bz.next_out = out.p + out.n;
            bz.avail_out = (unsigned)std::min<size_t>(out.cap - out.n, 1u << 30);
            const unsigned in0 = bz.avail_in, out0 = bz.avail_out;
            rc = step(&bz);
            pos += in0 - bz.avail_in;
            out.n += out0 - bz.avail_out;
            if (rc != 0 && rc != 4) { end(&bz); throw Error(SUFR_B200_ERR_IO, std::string(path) + ": corrupt bzip2 data"); }
            if (rc != 4 && pos >= n && in0 == bz.avail_in && out0 == bz.avail_out) {
                end(&bz);
                throw Error(SUFR_B200_ERR_IO, std::string(path) + ": truncated bzip2 data");
            }
        }
        end(&bz);
    }
}

void inflate_xz(const char* path, const char* src, size_t n, Inflated& out) {
    static const char* const names[] = {"liblzma.so.5", "liblzma.so", nullptr};
    void* lib = runtime_lib(path, names);
    // lzma_stream_buffer_decode(memlimit, flags, allocator, in, in_pos, in_size, out, out_pos, out_size)
    auto decode = runtime_sym<int (*)(uint64_t*, uint32_t, const void*, const uint8_t*, size_t*, size_t, uint8_t*, size_t*, size_t)>(
        lib, "lzma_stream_buffer_decode");
    size_t guess = n * 6 + (1u << 20);
    for (;;) {
        out.n = 0;
        out.need(guess);
        uint64_t memlimit = ~0ull;
        size_t in_pos = 0, out_pos = 0;
        const int rc = decode(&memlimit, 0x08 /* LZMA_CONCATENATED */, nullptr, (const uint8_t*)src, &in_pos, n, (uint8_t*)out.p,
                              &out_pos, out.cap);
        if (rc == 0) { out.n = out_pos; return; }
        // LZMA_BUF_ERROR (10) means "output too small" -- or, when output space is left, that the input ends early
        if (rc == 10 && out_pos < out.cap) throw Error(SUFR_B200_ERR_IO, std::string(path) + ": truncated xz data");
        if (rc != 10 || guess > (1ull << 40)) throw Error(SUFR_B200_ERR_IO, std::string(path) + ": corrupt xz data");
        guess *= 2;
    }
}

// replaces a compressed file image by its content
void maybe_decompress(const char* path, char*& p, size_t& n) {
    const unsigned char* u = (const unsigned char*)p;
    Inflated out;
    if (n >= 2 && u[0] == 0x1F && u[1] == 0x8B) inflate_gzip(path, p, n, out);
    else if (n >= 4 && u[0] == 0x28 && u[1] == 0xB5 && u[2] == 0x2F && u[3] == 0xFD) inflate_zstd(path, p, n, out);
    else if (n >= 3 && u[0] == 'B' && u[1] == 'Z' && u[2] == 'h') inflate_bzip2(path, p, n, out);
    else if (n >= 6 && u[0] == 0xFD && u[1] == '7' && u[2] == 'z' && u[3] == 'X' && u[4] == 'Z' && u[5] == 0) inflate_xz(path, p, n, out);
    else return;
    free(p);
    p = out.p;
    n = out.n;
}

void load_file_raw(const char* path, FileData& d);
void load_file(const char* path, FileData& d) {
    load_file_raw(path, d);
    maybe_decompress(path, d.p, d.n);
}

void load_file_raw(const char* path, FileData& d) {
    int fd = open(path, O_RDONLY);
    if (fd < 0) throw Error(SUFR_B200_ERR_IO, std::string(path) + ": " + strerror(errno));
    struct stat st;
    if (fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0) {
        d.n = (size_t)st.st_size;
        d.p = (char*)malloc(d.n);
        if (!d.p) { close(fd); throw Error(SUFR_B200_ERR_OUT_OF_MEMORY, std::string(path) + ": out of host memory"); }
        const int T = ingest_threads(d.n);
        try {
            parallel_for(T, [&](int t) {
                size_t lo = d.n * (size_t)t / T, hi = d.n * (size_t)(t + 1) / T;
                while (lo < hi) {
                    ssize_t got = pread(fd, d.p + lo, std::min<size_t>(hi - lo, 1u << 30), (off_t)lo);
                    if (got < 0 && errno == EINTR) continue;
                    if (got <= 0) throw Error(SUFR_B200_ERR_IO, std::string(path) + ": " + (got < 0 ? strerror(errno) : "short read"));
                    lo += (size_t)got;
                }
            });
        } catch (...) { close(fd); throw; }
        close(fd);
        return;
    }
    // pipes and other non-regular files: sequential read
    std::string data;
    char buf[1 << 16];
    ssize_t got;
    while ((got = read(fd, buf, sizeof(buf))) != 0) {
        if (got < 0) { if (errno == EINTR) continue; close(fd); throw Error(SUFR_B200_ERR_IO, std::string(path) + ": " + strerror(errno)); }
        data.append(buf, (size_t)got);
    }
    close(fd);
    d.n = data.size();
    d.p = (char*)malloc(std::max<size_t>(1, d.n));
    memcpy(d.p, data.data(), d.n);
}

// one line [b, e) starting at `pos` (e excludes "\n" and a "\r" right before it); advances pos behind the line
inline bool next_line(const char* data, size_t n, size_t& pos, size_t& b, size_t& e) {
    if (pos >= n) return false;
    b = pos;
    const void* nl = memchr(data + pos, '\n', n - pos);
    e = nl ? (size_t)((const char*)nl - data) : n;
    pos = e + 1;
    if (e > b && data[e - 1] == '\r') e--;
    return true;
}

std::string record_name(const char* data, size_t hb, size_t he, uint64_t ordinal) {  // util.rs:73-76
    size_t s = hb;
    while (s < he && isspace((unsigned char)data[s])) s++;
    size_t e = s;
    while (e < he && !isspace((unsigned char)data[e])) e++;
    return e > s ? std::string(data + s, e - s) : std::to_string(ordinal + 1);
}

struct Slice {
    size_t lo = 0, hi = 0;        // lines that START in [lo, hi)
    uint64_t seq_bytes = 0;       // sequence bytes of the slice
    uint64_t headers = 0;
    uint64_t out_off = 0;         // where the slice's output starts
    uint64_t first_record = 0;    // ordinal of the slice's first header
    std::vector<uint64_t> starts;
    std::vector<std::pair<size_t, size_t>> header_lines;
};

}  // namespace

void read_sequence_file(const char* path, uint8_t delim, SufrB200Sequences* out) {
    memset(out, 0, sizeof(*out));
    FileData file;
    load_file(path, file);
    const char* data = file.p;
    const size_t n = file.n;
    if (n == 0) throw Error(SUFR_B200_ERR_IO, std::string(path) + ": empty input (no FASTA/FASTQ record)");
    if (data[0] != '>' && data[0] != '@')
        throw Error(SUFR_B200_ERR_IO, std::string(path) + ": not a FASTA/FASTQ file");

    std::vector<uint64_t> starts;
    std::vector<std::string> names;
    uint8_t* seq = nullptr;
    uint64_t seq_len = 0;

    if (data[0] == '>') {
        const int T = ingest_threads(n);
        std::vector<Slice> sl(T);
        for (int t = 0; t < T; t++) {  // slice boundaries moved forward to the next line start
            size_t lo = n * (size_t)t / T;
            if (t > 0 && lo > 0 && data[lo - 1] != '\n') {
                const void* nl = memchr(data + lo, '\n', n - lo);
                lo = nl ? (size_t)((const char*)nl - data) + 1 : n;
            }
            sl[t].lo = lo;
            if (t > 0) sl[t - 1].hi = lo;
        }
        sl[T - 1].hi = n;
        for (int t = 1; t < T; t++) if (sl[t].lo < sl[t - 1].lo) sl[t].lo = sl[t - 1].lo;  // (monotone by construction)
        parallel_for(T, [&](int t) {  // pass 1: sizes
            Slice& c = sl[t];
            size_t pos = c.lo, b, e;
            while (pos < c.hi && next_line(data, n, pos, b, e)) {
                if (e > b && data[b] == '>') { c.headers++; c.header_lines.push_back({b + 1, e}); }
                else c.seq_bytes += e - b;
            }
        });
        uint64_t off = 0, rec = 0;
        for (int t = 0; t < T; t++) {
            sl[t].out_off = off;
            sl[t].first_record = rec;
            off += sl[t].seq_bytes + sl[t].headers;  // one delimiter per header ...
            rec += sl[t].headers;
        }
        seq_len = off - 1 + 1;  // ... except the first record (util.rs:62-64), plus the sentinel
        seq = (uint8_t*)malloc(seq_len);
        if (!seq) throw Error(SUFR_B200_ERR_OUT_OF_MEMORY, std::string(path) + ": out of host memory");
        parallel_for(T, [&](int t) {  // pass 2: write every slice at its final offset
            Slice& c = sl[t];
            // the global first header writes no delimiter, so everything behind it sits one byte earlier
            uint64_t o = c.out_off - (t > 0 ? 1 : 0);
            uint64_t ordinal = c.first_record;
            size_t pos = c.lo, b, e;
            while (pos < c.hi && next_line(data, n, pos, b, e)) {
                if (e > b && data[b] == '>') {
                    if (ordinal > 0) seq[o++] = delim;
                    c.starts.push_back(o);
                    ordinal++;
                } else {
                    memcpy(seq + o, data + b, e - b);
                    o += e - b;
                }
            }
        });
        seq[seq_len - 1] = '$';  // SENTINEL_CHARACTER, types.rs:20 / util.rs:82
        for (int t = 0; t < T; t++) {
            uint64_t ordinal = sl[t].first_record;
            for (size_t k = 0; k < sl[t].starts.size(); k++) {
                starts.push_back(sl[t].starts[k]);
                ordinal++;
                names.push_back(record_name(data, sl[t].header_lines[k].first, sl[t].header_lines[k].second, ordinal));
            }
        }
    } else {
        // FASTQ: four lines per record (header, sequence, '+' line, qualities)
        auto line_start = [&](size_t p) {  // first line start at or behind p
            if (p == 0 || p >= n || data[p - 1] == '\n') return std::min(p, n);
            const void* nl = memchr(data + p, '\n', n - p);
            return nl ? (size_t)((const char*)nl - data) + 1 : n;
        };
        auto is_record_start = [&](size_t p) {  // '@' line whose second successor is a '+' line
            if (p >= n || data[p] != '@') return false;
            size_t pos = p, b, e;
            if (!next_line(data, n, pos, b, e) || !next_line(data, n, pos, b, e)) return false;
            return pos < n && data[pos] == '+';
        };
        int T = ingest_threads(n);
        std::vector<Slice> sl(T);
        for (int t = 0; t < T; t++) {
            size_t lo = t == 0 ? 0 : line_start(n * (size_t)t / T);
            for (int tries = 0; t > 0 && lo < n && !is_record_start(lo) && tries < 8; tries++) {
                size_t pos = lo, b, e;
                next_line(data, n, pos, b, e);
                lo = pos;
            }
            if (t > 0 && lo < n && !is_record_start(lo)) lo = n;  // malformed neighbourhood: leave it to the slice before
            sl[t].lo = std::min(lo, n);
            if (t > 0) {
                if (sl[t].lo < sl[t - 1].lo) sl[t].lo = sl[t - 1].lo;
                sl[t - 1].hi = sl[t].lo;
            }
        }
        sl[T - 1].hi = n;
        parallel_for(T, [&](int t) {  // pass 1: sizes
            Slice& c = sl[t];
            size_t pos = c.lo, b, e;
            while (pos < c.hi && next_line(data, n, pos, b, e)) {
                if (e == b) continue;
                size_t sb, se, xb, xe;
                if (!next_line(data, n, pos, sb, se) || !next_line(data, n, pos, xb, xe) || !next_line(data, n, pos, xb, xe))
                    throw Error(SUFR_B200_ERR_IO, std::string(path) + ": truncated FASTQ record");
                c.headers++;
                c.header_lines.push_back({b + 1, e});
                c.seq_bytes += se - sb;
            }
        });
        uint64_t off = 0, rec = 0;
        for (int t = 0; t < T; t++) {
            sl[t].out_off = off;
            sl[t].first_record = rec;
            off += sl[t].seq_bytes + sl[t].headers;
            rec += sl[t].headers;
        }
        seq_len = rec ? off : 1;  // delimiters between records + the sentinel = one byte per record
        seq = (uint8_t*)malloc(seq_len);
        if (!seq) throw Error(SUFR_B200_ERR_OUT_OF_MEMORY, std::string(path) + ": out of host memory");
        parallel_for(T, [&](int t) {  // pass 2
            Slice& c = sl[t];
            uint64_t o = c.out_off - (c.first_record > 0 ? 1 : 0);
            uint64_t ordinal = c.first_record;
            size_t pos = c.lo, b, e;
            while (pos < c.hi && next_line(data, n, pos, b, e)) {
                if (e == b) continue;
                size_t sb = 0, se = 0, xb, xe;
                next_line(data, n, pos, sb, se);
                next_line(data, n, pos, xb, xe);
                next_line(data, n, pos, xb, xe);
                if (ordinal > 0) seq[o++] = delim;
                c.starts.push_back(o);
                ordinal++;
                memcpy(seq + o, data + sb, se - sb);
                o += se - sb;
            }
        });
        seq[seq_len - 1] = '$';
        for (int t = 0; t < T; t++) {
            uint64_t ordinal = sl[t].first_record;
            for (size_t k = 0; k < sl[t].starts.size(); k++) {
                starts.push_back(sl[t].starts[k]);
                ordinal++;
                names.push_back(record_name(data, sl[t].header_lines[k].first, sl[t].header_lines[k].second, ordinal));
            }
        }
    }

    out->seq_len = seq_len;
    out->seq = seq;
    out->num_sequences = starts.size();
    out->start_positions = (uint64_t*)malloc(std::max<size_t>(1, starts.size()) * 8);
    out->sequence_names = (char**)malloc(std::max<size_t>(1, names.size()) * sizeof(char*));
    for (size_t k = 0; k < starts.size(); k++) {
        out->start_positions[k] = starts[k];
        out->sequence_names[k] = strdup(names[k].c_str());
    }
}

void free_sequences(SufrB200Sequences* s) {
    if (!s) return;
    free(s->seq);
    free(s->start_positions);
    for (uint64_t k = 0; k < s->num_sequences; k++) free(s->sequence_names[k]);
    free(s->sequence_names);
    memset(s, 0, sizeof(*s));
}

}  // namespace sufr
