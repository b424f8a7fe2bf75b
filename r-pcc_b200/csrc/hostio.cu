// hostio.cu -- the host side of the batch tool as native threads (SURVEY 8(f) rank 2): reading KITTI .bin files
// straight into the pinned upload buffer, and the entropy-coder pool that turns the sections an encode call left in
// pinned host memory into `.rpcc` files.
//
// The reference does both per frame under the GIL: np.fromfile + a slice (dataset/dataset.py:57-70) and
// BasicCompressor.compress_dict + save_compressed_bitstream (utils/compress_utils.py:167-179,255-310) inside the
// ThreadPoolExecutor closure of tools/compress_datalist.py:91-141.  The format is unchanged -- bzip2 level 9, byte for
// byte what the system's libbz2 (the library CPython's bz2 module links) writes, whether libbz2 itself or this
// library's encoder (bz2enc.cu) produced it -- so the files are the reference's; what changes is that no Python runs
// per frame, that the pool works on batch k out of one set of pinned buffers while the GPU fills the other set with
// batch k+1, and that the slow part of libbz2 on this data (its block sort) is avoided where that pays.
//
// libbz2 ships without headers in this image: the two prototypes used are declared here and resolved with dlopen.
#include <dlfcn.h>
#include <errno.h>
#include <fcntl.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

#include <condition_variable>
#include <deque>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

using namespace rpcc;

namespace {

typedef int (*bz_compress_fn)(char* dest, unsigned* destLen, char* source, unsigned sourceLen, int blockSize100k,
                              int verbosity, int workFactor);
typedef int (*bz_decompress_fn)(char* dest, unsigned* destLen, char* source, unsigned sourceLen, int small, int verbosity);

struct Bz2 {
  void* handle = nullptr;
  bz_compress_fn compress = nullptr;
  bz_decompress_fn decompress = nullptr;
};

const Bz2* bz2lib() {
  static Bz2 lib;
  static std::once_flag once;
  std::call_once(once, [] {
    for (const char* name : {"libbz2.so.1.0", "libbz2.so.1", "libbz2.so"}) {
      void* h = dlopen(name, RTLD_NOW | RTLD_LOCAL);
      if (!h) continue;
      lib.compress = reinterpret_cast<bz_compress_fn>(dlsym(h, "BZ2_bzBuffToBuffCompress"));
      lib.decompress = reinterpret_cast<bz_decompress_fn>(dlsym(h, "BZ2_bzBuffToBuffDecompress"));
      if (lib.compress && lib.decompress) { lib.handle = h; return; }
      dlclose(h);
    }
  });
  return lib.handle ? &lib : nullptr;
}

// One frame of a submitted batch: where its sections lie (in the caller's pinned buffers) and where the file goes.
// Four or five geometry sections, then optionally the intensity section.
constexpr int kMaxSec = 6;
struct Job {
  const unsigned char* sec[kMaxSec];
  size_t len[kMaxSec];
  int nsec;
  int slot[kMaxSec];         // CoderStats slot of each section: the same kind of data in every file
  int wf[kMaxSec];           // libbz2 work factor per section (0 = library default)
  std::string path;          // empty: no file
  unsigned char* blob;       // optional in-memory copy of the file (capacity blob_cap)
  size_t blob_cap;
  uint32_t* bytes_out;       // file size
  int* status_out;           // RPCC_OK or an error code
  long long ticket;
};

struct Ticket { long long id; int remaining; int status; };

}  // namespace

struct rpcc_packer {
  std::vector<std::thread> threads;
  std::mutex mu;
  std::condition_variable cv_work, cv_done;
  std::deque<Job> queue;
  std::deque<Ticket> tickets;
  long long next_ticket = 1;
  int coder = 0;             // 0 = the cheaper of the two per section (measured), 1 = libbz2, 2 = this library's encoder
  bool stop = false;
  char err[256] = "";
};

namespace {

// Two coders write the same bytes: libbz2 (the call CPython's bz2.compress makes, level 9; the work factor only chooses
// when libbz2 gives up on its main sort, never the bytes) and this library's own encoder (bz2enc.cu: induced sorting
// instead of libbz2's block sort -- 3 to 5 times faster on label sequences, on a par on noisy residuals, behind on
// small inputs).  Which one is faster depends on the section and on the data, so every worker keeps, per section of the
// file, a running cost per byte of both and uses the cheaper one, probing the other now and then.  mode: 0 = that,
// 1 = libbz2 only, 2 = own encoder (libbz2 where it declines).
struct CoderStats {
  double cost[2][kMaxSec] = {};   // ns per byte, [coder][section slot]
  unsigned seen[kMaxSec] = {};
};

inline double now_ns() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return 1e9 * (double)ts.tv_sec + (double)ts.tv_nsec;
}

// `.rpcc` = per section [int32 length][entropy-coded bytes] (utils/compress_utils.py:167-179)
int pack_one(const Bz2* bz, const Job& j, std::vector<unsigned char>& out, std::vector<char>& tmp, CoderStats& st, int mode) {
  out.clear();
  for (int s = 0; s < j.nsec; ++s) {
    const size_t n = j.len[s];
    if (n > 0x7fffffffu) return RPCC_ERR_ARG;
    unsigned cap = (unsigned)(n + n / 100 + 600);    // bzlib manual: 1 % + 600 bytes always suffices
    if (tmp.size() < cap) tmp.resize(cap);
    unsigned got = cap;
    const int slot = j.slot[s];
    // mode 0: now and then a worker codes the section with BOTH coders (same input, so the two costs compare like with
    // like) and keeps the running costs; in between the cheaper one is used.  A worker's very first section is not a
    // probe: the own encoder grows its scratch buffers on that call, and a first probe taken cold sent the worker to
    // libbz2 for its next 255 frames (measured on 4096 files: 783 frames/s against 915 with the own encoder forced).
    // Probes: frames 1, 16, then every 256th.
    bool probe = false;
    int use = mode == 1 ? 1 : 0;                     // 0 = own, 1 = libbz2
    if (mode == 0) {
      const unsigned k = st.seen[slot]++;
      probe = (k == 1u || k == 16u || (k > 0u && (k & 255u) == 0u)) && n >= 512;
      use = st.cost[1][slot] < st.cost[0][slot] ? 1 : 0;
    }
    int rc = RPCC_BZ2_DECLINED;
    auto run_own = [&]() -> int {
      size_t got2 = 0;
      const int r = rpcc_bz2_compress(j.sec[s], n, reinterpret_cast<uint8_t*>(tmp.data()), cap, &got2);
      got = (unsigned)got2;
      return r;
    };
    auto run_lib = [&]() -> int {
      got = cap;
      return bz->compress(tmp.data(), &got, reinterpret_cast<char*>(const_cast<unsigned char*>(j.sec[s])), (unsigned)n, 9, 0, j.wf[s]) == 0 ? RPCC_OK : RPCC_ERR_ARG;
    };
    auto note = [&](int which, double t0) {
      const double c = (now_ns() - t0) / (double)n;
      double& e = st.cost[which][slot];
      e = e == 0 ? c : 0.5 * e + 0.5 * c;
    };
    if (probe) {
      double t0 = now_ns();
      rc = run_own();
      if (rc == RPCC_OK) note(0, t0); else if (rc != RPCC_BZ2_DECLINED) return rc;
      t0 = now_ns();
      const int r2 = run_lib();                      // (its output is the one kept: identical bytes either way)
      if (r2 != RPCC_OK) return r2;
      note(1, t0);
      if (rc == RPCC_BZ2_DECLINED) st.cost[0][slot] = 1e30;   // the own encoder leaves this kind of section to libbz2
      rc = RPCC_OK;
    } else {
      if (use == 0) {
        rc = run_own();
        if (rc != RPCC_OK && rc != RPCC_BZ2_DECLINED) return rc;
      }
      if (rc == RPCC_BZ2_DECLINED) rc = run_lib();
      if (rc != RPCC_OK) return rc;
    }
    const int32_t len32 = (int32_t)got;
    const size_t at = out.size();
    out.resize(at + 4 + got);
    memcpy(out.data() + at, &len32, 4);
    memcpy(out.data() + at + 4, tmp.data(), got);
  }
  return RPCC_OK;
}

int write_file(const std::string& path, const unsigned char* data, size_t n) {
  const int fd = open(path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
  if (fd < 0) return RPCC_ERR_ARG;
  size_t done = 0;
  while (done < n) {
    const ssize_t w = write(fd, data + done, n - done);
    if (w < 0) { if (errno == EINTR) continue; close(fd); return RPCC_ERR_ARG; }
    done += (size_t)w;
  }
  return close(fd) == 0 ? RPCC_OK : RPCC_ERR_ARG;
}

void worker(rpcc_packer* pk) {
  const Bz2* bz = bz2lib();
  std::vector<unsigned char> out;
  std::vector<char> tmp;
  CoderStats stats;
  for (;;) {
    Job j;
    {
      std::unique_lock<std::mutex> lk(pk->mu);
      pk->cv_work.wait(lk, [&] { return pk->stop || !pk->queue.empty(); });
      if (pk->queue.empty()) return;      // stop requested and nothing left
      j = std::move(pk->queue.front());
      pk->queue.pop_front();
    }
    int rc = bz ? pack_one(bz, j, out, tmp, stats, pk->coder) : RPCC_ERR_ARG;
    if (rc == RPCC_OK) {
      if (j.bytes_out) *j.bytes_out = (uint32_t)out.size();
      if (j.blob) {
        if (out.size() <= j.blob_cap) memcpy(j.blob, out.data(), out.size());
        else rc = RPCC_ERR_CAPACITY;
      }
      if (rc == RPCC_OK && !j.path.empty()) rc = write_file(j.path, out.data(), out.size());
    }
    if (j.status_out) *j.status_out = rc;
    {
      std::lock_guard<std::mutex> lk(pk->mu);
      for (Ticket& t : pk->tickets)
        if (t.id == j.ticket) {
          if (rc != RPCC_OK && t.status == RPCC_OK) {
            t.status = rc;
            snprintf(pk->err, sizeof(pk->err), "rpcc_packer: frame could not be coded or written (%s)",
                     j.path.empty() ? "in memory" : j.path.c_str());
          }
          --t.remaining;
          break;
        }
    }
    pk->cv_done.notify_all();
  }
}

}  // namespace

extern "C" int rpcc_packer_create(int threads, const char* method, rpcc_packer** out) {
  RPCC_REQUIRE(out && method, "null pointer");
  RPCC_REQUIRE(threads >= 1 && threads <= 1024, "threads must be in [1, 1024]");
  if (strcmp(method, "bzip2") != 0) {
    set_error("rpcc_packer_create: only bzip2 runs on the native pool (got '%s'); the other coders stay in Python", method);
    return RPCC_ERR_ARG;
  }
  if (!bz2lib()) { set_error("rpcc_packer_create: libbz2.so.1.0 could not be loaded"); return RPCC_ERR_ARG; }
  rpcc_packer* pk = new (std::nothrow) rpcc_packer();
  RPCC_REQUIRE(pk != nullptr, "out of host memory");
  if (const char* e = getenv("RPCC_BZ2_CODER")) pk->coder = !strcmp(e, "libbz2") ? 1 : !strcmp(e, "own") ? 2 : 0;
  for (int i = 0; i < threads; ++i) pk->threads.emplace_back(worker, pk);
  *out = pk;
  return RPCC_OK;
}

extern "C" void rpcc_packer_destroy(rpcc_packer* pk) {
  if (!pk) return;
  {
    std::lock_guard<std::mutex> lk(pk->mu);
    pk->stop = true;
  }
  pk->cv_work.notify_all();
  for (std::thread& t : pk->threads) t.join();
  delete pk;
}

extern "C" int rpcc_packer_submit(rpcc_packer* pk, int B, int K, int cbytes, int uniform, const rpcc_frame_result* results,
                                  const float* model, const uint8_t* contour_bits, const uint16_t* seq,
                                  const int16_t* symbols, const uint8_t* salience, const char* const* paths,
                                  uint32_t* bytes_out, int* status_out, uint8_t* blobs, size_t blob_stride,
                                  long long* ticket_out) {
  return rpcc_packer_submit_intensity(pk, B, K, cbytes, uniform, results, model, contour_bits, seq, symbols, salience, nullptr,
                                      paths, bytes_out, status_out, blobs, blob_stride, ticket_out);
}

extern "C" int rpcc_packer_submit_intensity(rpcc_packer* pk, int B, int K, int cbytes, int uniform,
                                            const rpcc_frame_result* results, const float* model,
                                            const uint8_t* contour_bits, const uint16_t* seq, const int16_t* symbols,
                                            const uint8_t* salience, const uint8_t* intensity, const char* const* paths,
                                            uint32_t* bytes_out, int* status_out, uint8_t* blobs, size_t blob_stride,
                                            long long* ticket_out) {
  RPCC_REQUIRE(pk && results && model && contour_bits && seq && symbols && ticket_out, "null pointer");
  RPCC_REQUIRE(uniform || salience, "non-uniform frames need the salience table");
  RPCC_REQUIRE(B >= 0 && K >= 2 && cbytes >= 1, "bad sizes");
  std::vector<Job> jobs((size_t)B);
  size_t sym_at = 0, seq_at = 0;
  for (int b = 0; b < B; ++b) {
    const rpcc_frame_result& r = results[b];
    Job& j = jobs[b];
    const size_t rows = r.model_rows < (uint32_t)K ? r.model_rows : (uint32_t)K;
    int s = 0;
    // utils/compress_utils.py:170-178: salience_level (non-uniform only), contour_map, idx_sequence, plane_param,
    // residual_quantized
    if (!uniform) { j.sec[s] = salience + (size_t)b * K; j.len[s] = rows; j.wf[s] = 0; ++s; }
    j.sec[s] = contour_bits + (size_t)b * cbytes; j.len[s] = (size_t)cbytes; j.wf[s] = 0; ++s;
    j.sec[s] = reinterpret_cast<const unsigned char*>(seq + seq_at); j.len[s] = (size_t)r.seq_count * 2;
    // long label sequences are what libbz2's main sort struggles with: send them to its fallback sort at once
    // (identical bytes, half the time; compress_utils.py _BZ2_WORK_FACTOR)
    j.wf[s] = j.len[s] >= 32768 ? 1 : 0; ++s;
    j.sec[s] = reinterpret_cast<const unsigned char*>(model + (size_t)b * K * 4); j.len[s] = rows * 16; j.wf[s] = 0; ++s;
    j.sec[s] = reinterpret_cast<const unsigned char*>(symbols + sym_at); j.len[s] = (size_t)r.sym_count * 2; j.wf[s] = 0; ++s;
    for (int q = 0; q < s; ++q) j.slot[q] = q + (5 - s);   // the last four sections line up whether or not salience leads
    if (intensity) { j.sec[s] = intensity + sym_at; j.len[s] = r.sym_count; j.wf[s] = 0; j.slot[s] = 5; ++s; }
    j.nsec = s;
    sym_at += r.sym_count;
    seq_at += r.seq_count;
    if (paths && paths[b]) j.path = paths[b];
    j.blob = blobs ? blobs + (size_t)b * blob_stride : nullptr;
    j.blob_cap = blob_stride;
    j.bytes_out = bytes_out ? bytes_out + b : nullptr;
    j.status_out = status_out ? status_out + b : nullptr;
  }
  {
    std::lock_guard<std::mutex> lk(pk->mu);
    const long long id = pk->next_ticket++;
    pk->tickets.push_back({id, B, RPCC_OK});
    for (Job& j : jobs) { j.ticket = id; pk->queue.push_back(std::move(j)); }
    *ticket_out = id;
  }
  pk->cv_work.notify_all();
  return RPCC_OK;
}

extern "C" int rpcc_packer_wait(rpcc_packer* pk, long long ticket) {
  RPCC_REQUIRE(pk, "null pointer");
  std::unique_lock<std::mutex> lk(pk->mu);
  for (;;) {
    auto it = pk->tickets.begin();
    for (; it != pk->tickets.end(); ++it) if (it->id == ticket) break;
    if (it == pk->tickets.end()) return RPCC_OK;          // unknown or already collected
    if (it->remaining == 0) {
      const int rc = it->status;
      pk->tickets.erase(it);
      if (rc != RPCC_OK) set_error("%s", pk->err);
      return rc;
    }
    pk->cv_done.wait(lk);
  }
}

// dataset/dataset.py:57-63 for a KITTI `.bin`: rows of (x, y, z, intensity) f32; the intensity is dropped while the rows
// are copied into `dst` (the pinned upload buffer), so 12 bytes per point cross the PCIe link instead of 16.
// Reads through a 1 MiB thread-local bounce buffer; *rows_out = points in the file (even when cap_rows is too small,
// in which case RPCC_ERR_CAPACITY is returned and nothing past cap_rows is written).
extern "C" int rpcc_read_bin_xyz(const char* path, float* dst, int64_t cap_rows, int64_t* rows_out) {
  RPCC_REQUIRE(path && dst && rows_out, "null pointer");
  const int fd = open(path, O_RDONLY);
  if (fd < 0) { set_error("rpcc_read_bin_xyz: cannot open %s: %s", path, strerror(errno)); return RPCC_ERR_ARG; }
  struct stat st;
  if (fstat(fd, &st) != 0 || (st.st_size % 16) != 0) {
    close(fd);
    set_error("rpcc_read_bin_xyz: %s is not a whole number of 16-byte rows", path);
    return RPCC_ERR_ARG;
  }
  const int64_t rows = (int64_t)(st.st_size / 16);
  *rows_out = rows;
  if (rows > cap_rows) { close(fd); set_error("rpcc_read_bin_xyz: %s has %lld rows, room for %lld", path, (long long)rows, (long long)cap_rows); return RPCC_ERR_CAPACITY; }
  constexpr size_t kChunkRows = 65536;
  static thread_local std::vector<float> bounce;
  if (bounce.size() < kChunkRows * 4) bounce.resize(kChunkRows * 4);
  int64_t done = 0;
  while (done < rows) {
    const size_t want = (size_t)((rows - done) < (int64_t)kChunkRows ? (rows - done) : (int64_t)kChunkRows) * 16;
    size_t got = 0;
    while (got < want) {
      const ssize_t r = read(fd, reinterpret_cast<char*>(bounce.data()) + got, want - got);
      if (r < 0) { if (errno == EINTR) continue; close(fd); set_error("rpcc_read_bin_xyz: read error on %s", path); return RPCC_ERR_ARG; }
      if (r == 0) { close(fd); set_error("rpcc_read_bin_xyz: %s shrank while being read", path); return RPCC_ERR_ARG; }
      got += (size_t)r;
    }
    const size_t n = want / 16;
    float* o = dst + (size_t)done * 3;
    const float* in = bounce.data();
    for (size_t i = 0; i < n; ++i) { o[3 * i] = in[4 * i]; o[3 * i + 1] = in[4 * i + 1]; o[3 * i + 2] = in[4 * i + 2]; }
    done += (int64_t)n;
  }
  close(fd);
  return RPCC_OK;
}

// The same keeping whole rows (x, y, z, intensity): the file goes straight into `dst`.
extern "C" int rpcc_read_bin_rows(const char* path, float* dst, int64_t cap_rows, int64_t* rows_out) {
  RPCC_REQUIRE(path && dst && rows_out, "null pointer");
  const int fd = open(path, O_RDONLY);
  if (fd < 0) { set_error("rpcc_read_bin_rows: cannot open %s: %s", path, strerror(errno)); return RPCC_ERR_ARG; }
  struct stat st;
  if (fstat(fd, &st) != 0 || (st.st_size % 16) != 0) {
    close(fd);
    set_error("rpcc_read_bin_rows: %s is not a whole number of 16-byte rows", path);
    return RPCC_ERR_ARG;
  }
  const int64_t rows = (int64_t)(st.st_size / 16);
  *rows_out = rows;
  if (rows > cap_rows) { close(fd); set_error("rpcc_read_bin_rows: %s has %lld rows, room for %lld", path, (long long)rows, (long long)cap_rows); return RPCC_ERR_CAPACITY; }
  const size_t want = (size_t)rows * 16;
  size_t got = 0;
  while (got < want) {
    const ssize_t r = read(fd, reinterpret_cast<char*>(dst) + got, want - got);
    if (r < 0) { if (errno == EINTR) continue; close(fd); set_error("rpcc_read_bin_rows: read error on %s", path); return RPCC_ERR_ARG; }
    if (r == 0) { close(fd); set_error("rpcc_read_bin_rows: %s shrank while being read", path); return RPCC_ERR_ARG; }
    got += (size_t)r;
  }
  close(fd);
  return RPCC_OK;
}

namespace {

// Inverse of the section coder for the decode tools: the first `nsec` sections of one `.rpcc` buffer decompressed back to
// back into `dst`, their lengths into sec_len[0 .. nsec).  Sections after them are not looked at.
int unpack_sections(const char* fn, const uint8_t* blob, size_t n, int nsec, const char* last, uint8_t* dst, size_t cap,
                    uint32_t* sec_len) {
  const Bz2* bz = bz2lib();
  if (!bz) { set_error("%s: libbz2.so.1.0 could not be loaded", fn); return RPCC_ERR_ARG; }
  size_t at = 0, out = 0;
  for (int s = 0; s < nsec; ++s) {
    if (at == n && s == nsec - 1) { set_error("%s: the file has no %s section", fn, last); return RPCC_ERR_ARG; }
    if (at + 4 > n) { set_error("%s: truncated stream", fn); return RPCC_ERR_ARG; }
    int32_t len;
    memcpy(&len, blob + at, 4);
    at += 4;
    if (len < 0 || at + (size_t)len > n) { set_error("%s: bad section length", fn); return RPCC_ERR_ARG; }
    unsigned got = (unsigned)((cap - out) > 0xffffffffu ? 0xffffffffu : (cap - out));
    // this library's decoder first (bz2dec.cu); what it declines -- and every error verdict -- is libbz2's
    static const bool own_first = !(getenv("RPCC_BZ2_DECODER") && !strcmp(getenv("RPCC_BZ2_DECODER"), "libbz2"));
    size_t got2 = 0;
    if (own_first && rpcc_bz2_decompress(blob + at, (size_t)len, dst + out, got, &got2) == RPCC_OK) {
      got = (unsigned)got2;
    } else {
      const int rc = bz->decompress(reinterpret_cast<char*>(dst + out), &got, reinterpret_cast<char*>(const_cast<uint8_t*>(blob + at)), (unsigned)len, 0, 0);
      if (rc != 0) { set_error("%s: section %d does not decode (libbz2 %d)", fn, s, rc); return rc == -8 ? RPCC_ERR_CAPACITY : RPCC_ERR_ARG; }
    }
    sec_len[s] = got;
    out += got;
    at += (size_t)len;
  }
  return RPCC_OK;
}

}  // namespace

// sec_len[5] receives the lengths in file order (nsec = 4 uniform, 5 non-uniform); a trailing intensity section is skipped.
extern "C" int rpcc_unpack_rpcc(const uint8_t* blob, size_t n, int uniform, uint8_t* dst, size_t cap, uint32_t* sec_len) {
  RPCC_REQUIRE(blob && dst && sec_len, "null pointer");
  const int nsec = uniform ? 4 : 5;
  const int rc = unpack_sections("rpcc_unpack_rpcc", blob, n, nsec, "residual_quantized", dst, cap, sec_len);
  if (rc != RPCC_OK) return rc;
  for (int s = nsec; s < 5; ++s) sec_len[s] = 0;
  return RPCC_OK;
}

// sec_len[6]: the geometry sections as rpcc_unpack_rpcc, the intensity section at index 5.
extern "C" int rpcc_unpack_rpcc_intensity(const uint8_t* blob, size_t n, int uniform, uint8_t* dst, size_t cap,
                                          uint32_t* sec_len) {
  RPCC_REQUIRE(blob && dst && sec_len, "null pointer");
  const int nsec = uniform ? 5 : 6;
  uint32_t len[6] = {0, 0, 0, 0, 0, 0};
  const int rc = unpack_sections("rpcc_unpack_rpcc_intensity", blob, n, nsec, "intensity", dst, cap, len);
  if (rc != RPCC_OK) return rc;
  for (int s = 0; s < 5; ++s) sec_len[s] = s < nsec - 1 ? len[s] : 0;
  sec_len[5] = len[nsec - 1];
  return RPCC_OK;
}
