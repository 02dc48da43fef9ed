// Thread-local error string, version and the optional kernel-timing table of the C ABI.
#include "common.cuh"
#include "profile.cuh"
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include <cstring>
#include <cstdlib>
#include <algorithm>

namespace msmd {
static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static bool g_prof = false;
static std::mutex g_prof_mu;
struct Pending { std::string name; cudaEvent_t e0, e1; };
static std::vector<Pending> g_pending;
static std::map<std::string, std::pair<double, long>> g_totals;

bool profiling_on() { return g_prof; }

ProfileScope::ProfileScope(const char* n, cudaStream_t s) : name(n), st(s) {
  if (!g_prof) return;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(s, &cs);
  if (cs != cudaStreamCaptureStatusNone) return;  // events inside a graph capture cannot be timed
  cudaEventCreate(&e0);
  cudaEventRecord(e0, st);
}
ProfileScope::~ProfileScope() {
  if (!e0) return;
  cudaEvent_t e1;
  cudaEventCreate(&e1);
  cudaEventRecord(e1, st);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_pending.push_back({name, e0, e1});
}
}  // namespace msmd

extern "C" const char* msmd_last_error(void) { return msmd::g_err; }
extern "C" const char* msmd_version(void) { return "msmd_b200 0.1 sm_100a"; }

extern "C" int msmd_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(msmd::g_prof_mu);
  msmd::g_prof = on != 0;
  return MSMD_OK;
}

extern "C" int msmd_profile_reset(void) {
  std::lock_guard<std::mutex> lk(msmd::g_prof_mu);
  for (auto& p : msmd::g_pending) { cudaEventDestroy(p.e0); cudaEventDestroy(p.e1); }
  msmd::g_pending.clear();
  msmd::g_totals.clear();
  return MSMD_OK;
}

// Synchronises the pending event pairs and returns total milliseconds / launch count for `name`.
extern "C" int msmd_profile_query(const char* name, double* total_ms, int64_t* launches) {
  std::lock_guard<std::mutex> lk(msmd::g_prof_mu);
  for (auto& p : msmd::g_pending) {
    float ms = 0.f;
    cudaEventSynchronize(p.e1);
    if (cudaEventElapsedTime(&ms, p.e0, p.e1) == cudaSuccess) {
      auto& t = msmd::g_totals[p.name];
      t.first += ms;
      t.second += 1;
    }
    cudaEventDestroy(p.e0);
    cudaEventDestroy(p.e1);
  }
  msmd::g_pending.clear();
  auto it = msmd::g_totals.find(name ? name : "");
  if (total_ms) *total_ms = it == msmd::g_totals.end() ? 0.0 : it->second.first;
  if (launches) *launches = it == msmd::g_totals.end() ? 0 : it->second.second;
  return MSMD_OK;
}

// Writes "name total_ms launches\n" lines for every kernel class seen since the last reset.
extern "C" int msmd_profile_dump(char* buf, int64_t cap) {
  msmd_profile_query("", nullptr, nullptr);   // drain pending events
  std::lock_guard<std::mutex> lk(msmd::g_prof_mu);
  std::string out;
  for (auto& kv : msmd::g_totals) {
    char line[256];
    snprintf(line, sizeof(line), "%s %.6f %ld\n", kv.first.c_str(), kv.second.first, kv.second.second);
    out += line;
  }
  if (buf && cap > 0) {
    const size_t n = std::min<size_t>(out.size(), (size_t)cap - 1);
    memcpy(buf, out.data(), n);
    buf[n] = 0;
  }
  return MSMD_OK;
}
