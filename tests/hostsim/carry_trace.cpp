// carry_trace.cpp -- TEST INFRASTRUCTURE ONLY.  The carry sanitizer of the host simulation: linked with hostsim.cpp built with
// -DFQ_HOSTSIM_CARRY (build_carry.sh -> libfq_hostsim_carry.so), it receives every carry primitive of arith.cuh with its call
// site, counts per site how often each carry value went in and came out, and checks three rules on every event:
//   dropped carry  an end op (addc, subc, madc_hi) whose exact result does not fit 32 bits: its carry or borrow is lost
//   lost carry     a start op (add_cc, sub_cc, mad_lo_cc) while the last carry written was 1 and no op has read it
//   stale read     a middle or end op with no carry written since the last end op: it reads a carry of another chain
// A site can be forced to a carry-in of 0 or 1 (the mutation check of tests/test_carry.py).  Single-threaded, as the simulation's
// entry points are.
#define FQ_HOSTSIM 1
#include "../../fourq_b200/csrc/arith.cuh"
#include <cstdio>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

namespace {

struct Site {
  const char* file; u32 line, col; int kind;
  u64 calls, cin[2], cout[2], dropped, lost, stale;
};

std::unordered_map<u64, Site> g_sites;
std::vector<const char*> g_files;             // file_name() pointers seen, index = file id
// chain state
bool g_open = false;                          // a carry was written since the last end op
bool g_unread = false;                        // the last carry written has not been read
u32 g_last = 0;                               // its value
Site* g_writer = nullptr;                     // the site that wrote it
// forced site: basename, line, column, carry-in
std::string g_force_file; u32 g_force_line = 0, g_force_col = 0, g_force_cin = 0; bool g_force = false;

const char* base_name(const char* path) {
  const char* b = strrchr(path, '/');
  return b ? b + 1 : path;
}

Site& site_of(int kind, const std::source_location& loc) {
  const char* f = loc.file_name();
  u64 id = 0;
  while (id < g_files.size() && g_files[id] != f) id++;
  if (id == g_files.size()) g_files.push_back(f);
  const u64 key = (id << 48) | ((u64)loc.line() << 16) | loc.column();
  auto it = g_sites.find(key);
  if (it == g_sites.end()) {
    Site s = {};
    s.file = base_name(f); s.line = loc.line(); s.col = loc.column(); s.kind = kind;
    it = g_sites.emplace(key, s).first;
  }
  return it->second;
}

}  // namespace

namespace fqsim {
u32 carry_event(CarryKind kind, u32 cin, u64 exact0, const std::source_location& loc) {
  Site& s = site_of(kind, loc);
  const bool start = kind <= CK_MAD_LO_CC, end = kind >= CK_ADDC;
  const bool sub = kind == CK_SUB_CC || kind == CK_SUBC_CC || kind == CK_SUBC;
  if (!start && g_force && loc.line() == g_force_line && loc.column() == g_force_col && g_force_file == s.file) cin = g_force_cin;
  const u64 exact = (sub ? exact0 - cin : exact0 + cin) & 0x1ffffffffull;      // 33 bits: bit 32 = carry (borrow) out
  const u32 out = (u32)(exact >> 32);
  s.calls++;
  if (start) {
    if (g_unread && g_last == 1) { s.lost++; if (g_writer) g_writer->lost++; }
  } else {
    s.cin[cin]++;
    if (!g_open) s.stale++;
  }
  if (end) {
    if (out) s.dropped++;
    g_open = false; g_unread = false;
  } else {
    s.cout[out]++;
    g_open = true; g_unread = true; g_last = out; g_writer = &s;
  }
  return cin;
}
}  // namespace fqsim

extern "C" {

// clears the counters and the chain state (a forced site stays)
void carry_reset() {
  g_sites.clear();
  g_open = g_unread = false; g_last = 0; g_writer = nullptr;
}

// one line per site executed since the last reset: file line column kind calls cin0 cin1 cout0 cout1 dropped lost stale,
// tab-separated.  Writes at most cap bytes (NUL-terminated) and returns the length the whole table needs.
size_t carry_dump(char* buf, size_t cap) {
  std::string t;
  char line[512];
  for (const auto& kv : g_sites) {
    const Site& s = kv.second;
    snprintf(line, sizeof line, "%s\t%u\t%u\t%d\t%llu\t%llu\t%llu\t%llu\t%llu\t%llu\t%llu\t%llu\n", s.file, s.line, s.col, s.kind,
             (unsigned long long)s.calls, (unsigned long long)s.cin[0], (unsigned long long)s.cin[1], (unsigned long long)s.cout[0],
             (unsigned long long)s.cout[1], (unsigned long long)s.dropped, (unsigned long long)s.lost, (unsigned long long)s.stale);
    t += line;
  }
  if (buf && cap) { size_t m = t.size() < cap - 1 ? t.size() : cap - 1; memcpy(buf, t.data(), m); buf[m] = 0; }
  return t.size() + 1;
}

// forces the carry-in of the middle or end op at file (base name), line, column to cin (0 or 1); cin < 0 clears the force
void carry_force_site(const char* file, int line, int col, int cin) {
  g_force = cin >= 0;
  g_force_file = file ? file : ""; g_force_line = (u32)line; g_force_col = (u32)col; g_force_cin = (u32)(cin > 0);
}

}  // extern "C"
