// sharded.cpp — ugx_sharded_*: ONE process, several GPUs (SURVEY.md 8e).  The corpus is cut into one line-aligned
// shard per device (forward from n*r/N to the next newline, so a line belongs to exactly one shard and no halo is
// needed); a host thread per device drives that device's pattern + scanner through the same C ABI a single-GPU
// caller uses; the only exchange of the path — per-shard {matches, newlines} -> totals, record and line-number
// bases — goes through host memory: this call owns every device and already synchronises on each of them, so the
// 16 bytes per shard are summed on the host rather than all-gathered over NCCL (which would need a communicator and
// a stream sync for the same 16 bytes; the multi-PROCESS form, one rank per GPU, does use NCCL: ugrep_b200/sharding.py).
// This replaces the reference's file-level job queue (GrepMaster / GrepWorker, src/ugrep.cpp:4118-4432) for the case of
// one large input.
#include <cstring>
#include <functional>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/ugrep_b200.h"

struct ugx_sharded {
  std::vector<int> devices;
  std::vector<ugx_pattern*> patterns;
  std::vector<ugx_scanner*> scanners;
  std::vector<uint8_t*> dbuf;     // records mode: the shard on its device
  std::vector<uint64_t> dcap;
  bool pin = false;               // page-lock the caller's buffer for the duration of a scan
};

namespace {

thread_local std::string s_err;

int sfail(int code, const std::string& m)
{
  s_err = m;
  return code;
}

void cut_points(const uint8_t* buf, uint64_t n, int nshard, std::vector<uint64_t>& cuts)
{
  cuts.assign(1, 0);
  for (int r = 1; r < nshard; ++r)
  {
    uint64_t target = n / nshard * r + (n % nshard) * r / nshard;
    if (target < cuts.back())
      target = cuts.back();
    if (target >= n)
    {
      cuts.push_back(n);
      continue;
    }
    if (target == 0 || buf[target - 1] == '\n')
    {
      cuts.push_back(target);
      continue;
    }
    const void* q = memchr(buf + target, '\n', n - target);
    cuts.push_back(q != nullptr ? static_cast<uint64_t>(static_cast<const uint8_t*>(q) - buf) + 1 : n);
  }
  cuts.push_back(n);
}

} // namespace

extern "C" {

const char* ugx_sharded_last_error(void) { return s_err.c_str(); }

int ugx_sharded_create(const uint32_t* opc, uint32_t nop, const ugx_prefilter* pf, uint32_t matcher_flags, const int* devices,
                       int ndev, ugx_sharded** out)
{
  if (opc == nullptr || pf == nullptr || devices == nullptr || ndev < 1 || ndev > 64 || out == nullptr)
    return sfail(UGX_E_INVALID, "ugx_sharded_create: bad argument");
  ugx_sharded* s = new (std::nothrow) ugx_sharded();
  if (s == nullptr)
    return sfail(UGX_E_NOMEM, "out of host memory");
  for (int i = 0; i < ndev; ++i)
  {
    ugx_pattern* p = nullptr;
    ugx_scanner* sc = nullptr;
    int rc = ugx_pattern_create(opc, nop, pf, matcher_flags, devices[i], &p);
    if (rc == UGX_OK)
      rc = ugx_scanner_create(devices[i], nullptr, &sc);
    if (rc != UGX_OK)
    {
      const std::string why = ugx_last_error();
      if (p != nullptr)
        ugx_pattern_destroy(p);
      ugx_sharded_destroy(s);
      return sfail(rc, why);
    }
    s->devices.push_back(devices[i]);
    s->patterns.push_back(p);
    s->scanners.push_back(sc);
    s->dbuf.push_back(nullptr);
    s->dcap.push_back(0);
  }
  *out = s;
  return UGX_OK;
}

void ugx_sharded_destroy(ugx_sharded* s)
{
  if (s == nullptr)
    return;
  for (size_t i = 0; i < s->scanners.size(); ++i)
  {
    ugx_scanner_destroy(s->scanners[i]);
    ugx_pattern_destroy(s->patterns[i]);
    if (s->dbuf[i] != nullptr)
    {
      cudaSetDevice(s->devices[i]);
      cudaFree(s->dbuf[i]);
    }
  }
  delete s;
}

int ugx_sharded_set_option(ugx_sharded* s, const char* name, int value)
{
  if (s == nullptr || name == nullptr)
    return sfail(UGX_E_INVALID, "null argument");
  if (strcmp(name, "pin") == 0)
  {
    s->pin = value != 0;
    return UGX_OK;
  }
  for (ugx_scanner* sc : s->scanners)
  {
    const int rc = ugx_scanner_set_option(sc, name, value);
    if (rc != UGX_OK)
      return sfail(rc, ugx_last_error());
  }
  return UGX_OK;
}

} // extern "C"

namespace {

// ugx_sharded_scan, and with `lines` ugx_sharded_find_lines (mode UGX_MODE_RECORDS, out is a ugx_line array): line
// records go through the same two phases as match records, with ugx_find_lines_device in place of ugx_find_all_device
int sharded_run(ugx_sharded* s, const void* host_buf, uint64_t n, int mode, bool lines, uint32_t lflags, void* out,
                uint64_t cap, uint64_t* n_out, ugx_totals* totals, ugx_shard* shards)
{
  if (s == nullptr || (host_buf == nullptr && n != 0) || mode < UGX_MODE_LINES || mode > UGX_MODE_RECORDS)
    return sfail(UGX_E_INVALID, "ugx_sharded_scan: bad argument");
  const int nd = static_cast<int>(s->scanners.size());
  const uint8_t* buf = static_cast<const uint8_t*>(host_buf);
  std::vector<uint64_t> cuts;
  cut_points(buf, n, nd, cuts);
  bool pinned = false;
  if (s->pin && n > 0)
    pinned = cudaHostRegister(const_cast<void*>(host_buf), n, cudaHostRegisterPortable | cudaHostRegisterReadOnly) == cudaSuccess;
  if (!pinned)
    cudaGetLastError();
  std::vector<ugx_totals> tt(nd);
  std::vector<int> rcs(nd, UGX_OK);
  std::vector<std::string> errs(nd);
  std::vector<uint64_t> nrec(nd, 0);
  auto each = [&](const std::function<void(int)>& f) {
    std::vector<std::thread> th;
    for (int r = 0; r < nd; ++r)
      th.emplace_back([&, r]() { f(r); });
    for (auto& t : th)
      t.join();
  };
  const bool records = mode == UGX_MODE_RECORDS;
  // ---- phase 1: every device scans its shard.  Records need the line-number bases first, i.e. the newline counts of
  // the shards before: the shard goes to its device once, is counted there, then scanned with its bases.
  each([&](int r) {
    memset(&tt[r], 0, sizeof(ugx_totals));
    const uint64_t len = cuts[r + 1] - cuts[r];
    if (len == 0)
      return;
    if (!records)
    {
      rcs[r] = mode == UGX_MODE_LINES ? ugx_count_lines(s->scanners[r], s->patterns[r], buf + cuts[r], len, &tt[r])
                                      : ugx_count_matches(s->scanners[r], s->patterns[r], buf + cuts[r], len, &tt[r]);
      if (rcs[r] == UGX_OK && (tt[r].flags & UGX_TOT_NEWLINES) == 0)
      {
        // the streaming `-c` kernels only count newlines on request: the bases of later shards want them
        ugx_totals nl;
        rcs[r] = ugx_count_newlines(s->scanners[r], buf + cuts[r], len, &nl);
        tt[r].newlines = nl.newlines;
      }
    }
    else
    {
      cudaError_t e = cudaSetDevice(s->devices[r]);
      if (e == cudaSuccess && s->dcap[r] < len + 16)
      {
        if (s->dbuf[r] != nullptr)
          cudaFree(s->dbuf[r]);
        s->dbuf[r] = nullptr;
        s->dcap[r] = 0;
        e = cudaMalloc(reinterpret_cast<void**>(&s->dbuf[r]), len + len / 8 + 16);
        if (e == cudaSuccess)
          s->dcap[r] = len + len / 8 + 16;
      }
      if (e == cudaSuccess)
        e = cudaMemcpy(s->dbuf[r], buf + cuts[r], len, cudaMemcpyHostToDevice);
      if (e != cudaSuccess)
      {
        rcs[r] = UGX_E_CUDA;
        errs[r] = cudaGetErrorString(e);
        return;
      }
      rcs[r] = ugx_count_newlines(s->scanners[r], s->dbuf[r], len, &tt[r]);
    }
    if (rcs[r] != UGX_OK && errs[r].empty())
      errs[r] = ugx_last_error();
  });
  int rc = UGX_OK;
  for (int r = 0; r < nd && rc == UGX_OK; ++r)
    if (rcs[r] != UGX_OK)
      rc = sfail(rcs[r], "shard " + std::to_string(r) + ": " + errs[r]);
  // ---- the exchange: bases from the per-shard counts (host sum; see the file header)
  std::vector<uint64_t> line_base(nd + 1, 0);
  for (int r = 0; r < nd; ++r)
    line_base[r + 1] = line_base[r] + tt[r].newlines;
  if (rc == UGX_OK && records)
  {
    each([&](int r) {
      const uint64_t len = cuts[r + 1] - cuts[r];
      if (len == 0)
        return;
      ugx_totals t2;
      if (lines)
      {
        const ugx_line* dev = nullptr;
        rcs[r] = ugx_find_lines_device(s->scanners[r], s->patterns[r], s->dbuf[r], len, cuts[r], line_base[r], lflags, &dev,
                                       &nrec[r], &t2);
      }
      else
      {
        const ugx_match* dev = nullptr;
        rcs[r] = ugx_find_all_device(s->scanners[r], s->patterns[r], s->dbuf[r], len, cuts[r], line_base[r], &dev, &nrec[r], &t2);
      }
      if (rcs[r] != UGX_OK)
        errs[r] = ugx_last_error();
      else
      {
        t2.kernel_ms += tt[r].kernel_ms;
        t2.launches += tt[r].launches;
        tt[r] = t2;
      }
    });
    for (int r = 0; r < nd && rc == UGX_OK; ++r)
      if (rcs[r] != UGX_OK)
        rc = sfail(rcs[r], "shard " + std::to_string(r) + ": " + errs[r]);
  }
  std::vector<uint64_t> rec_base(nd + 1, 0);
  for (int r = 0; r < nd; ++r)
    rec_base[r + 1] = rec_base[r] + (records ? nrec[r] : tt[r].matches);
  if (rc == UGX_OK && records)
  {
    if (n_out != nullptr)
      *n_out = rec_base[nd];
    if (rec_base[nd] > cap)
      rc = sfail(UGX_E_OVERFLOW, "record buffer too small");
    else if (rec_base[nd] > 0 && out == nullptr)
      rc = sfail(UGX_E_INVALID, "null record buffer");
    else
    {
      // records come back in shard order = input order; offsets and line numbers already carry their bases
      each([&](int r) {
        if (nrec[r] != 0)
          rcs[r] = lines ? ugx_scanner_fetch_lines(s->scanners[r], static_cast<ugx_line*>(out) + rec_base[r], 0, nrec[r])
                         : ugx_scanner_fetch(s->scanners[r], static_cast<ugx_match*>(out) + rec_base[r], 0, nrec[r]);
        if (rcs[r] != UGX_OK)
          errs[r] = ugx_last_error();
      });
      for (int r = 0; r < nd && rc == UGX_OK; ++r)
        if (rcs[r] != UGX_OK)
          rc = sfail(rcs[r], "shard " + std::to_string(r) + ": " + errs[r]);
    }
  }
  else if (n_out != nullptr)
    *n_out = 0;
  if (pinned)
    cudaHostUnregister(const_cast<void*>(host_buf));
  if (rc != UGX_OK)
    return rc;
  if (totals != nullptr)
  {
    memset(totals, 0, sizeof(*totals));
    totals->flags = UGX_TOT_NEWLINES;
    for (int r = 0; r < nd; ++r)
    {
      totals->matches += tt[r].matches;
      totals->newlines += tt[r].newlines;
      totals->flags |= tt[r].flags & UGX_TOT_SPAN_HANDOVER;
      totals->launches += tt[r].launches;
      if (tt[r].kernel_ms > totals->kernel_ms)
        totals->kernel_ms = tt[r].kernel_ms; // the devices run side by side: the slowest one
      if (tt[r].kernel != UGX_K_NONE)
        totals->kernel = tt[r].kernel;
    }
  }
  if (shards != nullptr)
    for (int r = 0; r < nd; ++r)
    {
      shards[r].device = s->devices[r];
      shards[r].begin = cuts[r];
      shards[r].end = cuts[r + 1];
      shards[r].matches = tt[r].matches;
      shards[r].newlines = tt[r].newlines;
      shards[r].line_base = line_base[r];
      shards[r].record_base = rec_base[r];
      shards[r].kernel_ms = tt[r].kernel_ms;
    }
  return UGX_OK;
}

} // namespace

extern "C" {

int ugx_sharded_scan(ugx_sharded* s, const void* host_buf, uint64_t n, int mode, ugx_match* out, uint64_t cap,
                     uint64_t* n_out, ugx_totals* totals, ugx_shard* shards)
{
  return sharded_run(s, host_buf, n, mode, false, 0, out, cap, n_out, totals, shards);
}

int ugx_sharded_find_lines(ugx_sharded* s, const void* host_buf, uint64_t n, uint32_t flags, ugx_line* out, uint64_t cap,
                           uint64_t* n_out, ugx_totals* totals, ugx_shard* shards)
{
  if ((flags & ~UGX_LINES_INVERT) != 0)
    return sfail(UGX_E_INVALID, "ugx_sharded_find_lines: unknown flags");
  return sharded_run(s, host_buf, n, UGX_MODE_RECORDS, true, flags, out, cap, n_out, totals, shards);
}

} // extern "C"
