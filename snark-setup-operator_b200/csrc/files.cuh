// File plumbing of the `_file` entry points (SURVEY.md §8b, §8f.1): the reference CLI mmaps its inputs and creates its
// outputs with create_new; here inputs are mapped read-only (the H2D copies read straight from the page cache, piece by
// piece), outputs are created under a temporary name, mapped, filled by the D2H copies and renamed into place only when
// the call succeeded — a failed call never leaves a partial output (SURVEY.md §5), and an existing output is an error.
#pragma once
#include <sys/mman.h>
#include <sys/stat.h>
#include <fcntl.h>
#include <unistd.h>
#include <deque>
#include <string>
#include <mutex>
#include <vector>

#include "blake2b.h"

namespace sso {

// create_new on the final name: an output that already exists is an error
inline int refuse_existing(const char* fn, char* err, size_t errcap) {
  struct stat st;
  if (stat(fn, &st) == 0) { set_err(err, errcap, "cannot create %s (outputs must not exist)", fn); return SSO_E_IO; }
  return SSO_OK;
}

struct MappedFile {
  uint8_t* p = nullptr;
  size_t len = 0;
  int fd = -1;
  std::string path, tmp;
  bool output = false, owner = false, committed = false;

  MappedFile() = default;
  MappedFile(const MappedFile&) = delete;
  MappedFile& operator=(const MappedFile&) = delete;

  int open_ro(const char* fn, char* err, size_t errcap) {
    path = fn;
    fd = ::open(fn, O_RDONLY);
    if (fd < 0) { set_err(err, errcap, "cannot open %s", fn); return SSO_E_IO; }
    struct stat st;
    if (fstat(fd, &st) != 0) { set_err(err, errcap, "cannot stat %s", fn); return SSO_E_IO; }
    len = (size_t)st.st_size;
    if (len == 0) return SSO_OK;
    void* m = mmap(nullptr, len, PROT_READ, MAP_SHARED, fd, 0);
    if (m == MAP_FAILED) { set_err(err, errcap, "cannot map %s", fn); return SSO_E_IO; }
    p = (uint8_t*)m;
    madvise(p, len, MADV_SEQUENTIAL);
    return SSO_OK;
  }
  // `owner` creates <fn>.sso-partial (create_new semantics on both names); a non-owner (another rank of the process group,
  // after the owner's barrier) opens the partial file the owner made
  int create(const char* fn, size_t size, bool is_owner, char* err, size_t errcap) {
    path = fn;
    tmp = path + ".sso-partial";
    output = true;
    owner = is_owner;
    len = size;
    if (owner) {
      int rc = refuse_existing(fn, err, errcap);
      if (rc) return rc;
      fd = ::open(tmp.c_str(), O_RDWR | O_CREAT | O_EXCL, 0644);
      if (fd < 0) { set_err(err, errcap, "cannot create %s (outputs must not exist)", tmp.c_str()); return SSO_E_IO; }
      if (ftruncate(fd, (off_t)size) != 0) { set_err(err, errcap, "cannot size %s to %zu bytes", tmp.c_str(), size); return SSO_E_IO; }
    } else {
      fd = ::open(tmp.c_str(), O_RDWR);
      if (fd < 0) { set_err(err, errcap, "cannot open %s", tmp.c_str()); return SSO_E_IO; }
    }
    void* m = mmap(nullptr, size, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    if (m == MAP_FAILED) { set_err(err, errcap, "cannot map %s", tmp.c_str()); return SSO_E_IO; }
    p = (uint8_t*)m;
    return SSO_OK;
  }
  void unmap() {
    if (p) { munmap(p, len); p = nullptr; }
    if (fd >= 0) { ::close(fd); fd = -1; }
  }
  // the call succeeded: the partial file takes its final name
  int commit(char* err, size_t errcap) {
    unmap();
    if (output && owner) {
      if (rename(tmp.c_str(), path.c_str()) != 0) { set_err(err, errcap, "cannot rename %s to %s", tmp.c_str(), path.c_str()); return SSO_E_IO; }
    }
    committed = true;
    return SSO_OK;
  }
  ~MappedFile() {
    unmap();
    if (output && owner && !committed) unlink(tmp.c_str());
  }
};

// Page-locked staging buffers for the chunk-sized file calls, cached across calls (cudaHostAlloc of 31 MB costs milliseconds;
// a pageable source makes cudaMemcpyAsync stage synchronously through the driver's own bounce buffers and serialises the
// lanes).  A lane takes a buffer, read()s the file into it — the H2D copy then runs at link speed beside the Blake2b of the same
// bytes —, and hands it back.
struct PinnedBuf { uint8_t* p = nullptr; size_t cap = 0; };
struct PinnedPool {
  std::mutex mu;
  std::vector<PinnedBuf> free_list;
  static PinnedPool& get() { static PinnedPool pool; return pool; }
  PinnedBuf take(size_t bytes) {
    {
      std::lock_guard<std::mutex> g(mu);
      for (size_t i = 0; i < free_list.size(); i++)
        if (free_list[i].cap >= bytes && free_list[i].cap <= 2 * bytes + (1u << 20)) { PinnedBuf b = free_list[i]; free_list.erase(free_list.begin() + i); return b; }
    }
    PinnedBuf b;
    if (cudaHostAlloc((void**)&b.p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); b.p = nullptr; return b; }
    b.cap = bytes;
    return b;
  }
  void give(PinnedBuf b) {
    if (!b.p) return;
    std::lock_guard<std::mutex> g(mu);
    if (free_list.size() >= 24) { cudaFreeHost(b.p); return; }
    free_list.push_back(b);
  }
};
struct PinnedLease {
  PinnedBuf b;
  explicit PinnedLease(size_t bytes) : b(PinnedPool::get().take(bytes)) {}
  ~PinnedLease() { PinnedPool::get().give(b); }
  PinnedLease(const PinnedLease&) = delete;
  PinnedLease& operator=(const PinnedLease&) = delete;
};
inline int read_file_into(const char* path, uint8_t* dst, size_t expect, char* err, size_t errcap) {
  int fd = ::open(path, O_RDONLY);
  if (fd < 0) { set_err(err, errcap, "cannot open %s", path); return SSO_E_IO; }
  struct stat st;
  if (fstat(fd, &st) != 0) { ::close(fd); set_err(err, errcap, "cannot stat %s", path); return SSO_E_IO; }
  if ((size_t)st.st_size != expect) { ::close(fd); set_err(err, errcap, "The size of %s should be correct: %zu != %zu", path, (size_t)st.st_size, expect); return SSO_E_ARG; }
  size_t got = 0;
  while (got < expect) {
    ssize_t r = read(fd, dst + got, expect - got);
    if (r <= 0) { ::close(fd); set_err(err, errcap, "short read on %s", path); return SSO_E_IO; }
    got += (size_t)r;
  }
  ::close(fd);
  return SSO_OK;
}

// Every output of one file call.  Each is created under <name>.sso-partial (create_new semantics on both names): the mapped
// outputs the call fills in place, and the small files written whole (the hash files; in the chunk-sized paths also the
// response or new challenge).  commit() renames them into place, mapped outputs first, then the small files in the order
// they were written; whatever is not committed is removed on destruction.  A mapped output created by a non-owner (another
// rank of the process group mapping the owner's partial file) is only detached from: never renamed, never removed.
struct Outputs {
  std::deque<MappedFile> mapped;
  std::vector<std::string> small;                // final names
  bool committed = false;

  Outputs() = default;
  Outputs(const Outputs&) = delete;
  Outputs& operator=(const Outputs&) = delete;

  int create_mapped(const char* fn, size_t size, bool owner, uint8_t** p, char* err, size_t errcap) {
    mapped.emplace_back();
    int rc = mapped.back().create(fn, size, owner, err, errcap);
    *p = mapped.back().p;
    return rc;
  }
  int write_whole(const char* fn, const uint8_t* data, size_t len, char* err, size_t errcap) {
    int rc = refuse_existing(fn, err, errcap);
    if (rc) return rc;
    const std::string tmp = std::string(fn) + ".sso-partial";
    int fd = ::open(tmp.c_str(), O_WRONLY | O_CREAT | O_EXCL, 0644);
    if (fd < 0) { set_err(err, errcap, "cannot create %s (outputs must not exist)", tmp.c_str()); return SSO_E_IO; }
    size_t put = 0;
    while (put < len) {
      ssize_t w = write(fd, data + put, len - put);
      if (w <= 0) { ::close(fd); unlink(tmp.c_str()); set_err(err, errcap, "short write on %s", tmp.c_str()); return SSO_E_IO; }
      put += (size_t)w;
    }
    ::close(fd);
    small.push_back(fn);
    return SSO_OK;
  }
  // the 64 raw bytes of Blake2b-512(data)
  int write_hash(const char* fn, const uint8_t* data, size_t len, char* err, size_t errcap) {
    uint8_t h[64];
    blake2b_512(data, len, h);
    return write_whole(fn, h, 64, err, errcap);
  }
  int commit(char* err, size_t errcap) {
    int rc;
    for (MappedFile& m : mapped)
      if ((rc = m.commit(err, errcap))) return rc;
    for (const std::string& fn : small) {
      const std::string tmp = fn + ".sso-partial";
      if (rename(tmp.c_str(), fn.c_str()) != 0) { set_err(err, errcap, "cannot rename %s to %s", tmp.c_str(), fn.c_str()); return SSO_E_IO; }
    }
    committed = true;
    return SSO_OK;
  }
  ~Outputs() {
    if (!committed)
      for (const std::string& fn : small) unlink((fn + ".sso-partial").c_str());
  }
};

}  // namespace sso
