// Test-only host build of icikt_owned.h.  The memory calls are wrapped at link time (-Wl,--wrap=...): an allocation
// returns a fresh fake address, or fails on request, and every free is checked against the live allocations.  So the
// array handles' ownership is checked without a device.  Streams and events go to the CUDA runtime itself.
// Prints "ok" and exits with 0, or names the first failed check and exits with 1.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <set>
#include <utility>

#include "../icikendalltau_b200/csrc/icikt_owned.h"

using icikt::DeviceArray;
using icikt::Event;
using icikt::PinnedArray;
using icikt::Stream;

namespace {

bool g_fail = false;       // the next allocations fail
int g_allocs = 0;          // allocation calls made
int g_bad_frees = 0;       // frees of an address that is not live
std::set<void*> g_live;    // allocated and not freed
uintptr_t g_next = 0x10000;

cudaError_t fake_alloc(void** p) {
  ++g_allocs;
  if (g_fail) return cudaErrorMemoryAllocation;
  *p = reinterpret_cast<void*>(g_next += 0x1000);
  g_live.insert(*p);
  return cudaSuccess;
}

cudaError_t fake_free(void* p) {
  if (!g_live.erase(p)) ++g_bad_frees;
  return cudaSuccess;
}

void check(bool ok, const char* what) {
  if (ok) return;
  std::printf("failed: %s\n", what);
  std::exit(1);
}

template <class A>
void check_array() {
  {
    A a;
    check(!a && a.get() == nullptr && a.size() == 0, "a new handle is empty");
    check(a.reserve(0) == cudaSuccess && a && a.size() == 1, "reserve(0) allocates one element");
    check(a.reserve(10) == cudaSuccess && a.size() == 10 && g_live.size() == 1, "reserve grows and frees the old");
    void* const held = a.get();
    const int allocs = g_allocs;
    check(a.reserve(10) == cudaSuccess && a.reserve(3) == cudaSuccess && a.get() == held && a.size() == 10 &&
              g_allocs == allocs,
          "reserve keeps an allocation that holds n");

    g_fail = true;
    check(a.reserve(11) == cudaErrorMemoryAllocation, "a failed reserve returns the error");
    check(!a && a.get() == nullptr && a.size() == 0 && g_live.empty(), "a failed reserve leaves the handle empty");
    check(a.reserve(1) == cudaErrorMemoryAllocation && g_allocs == allocs + 2, "the next reserve tries again");
    g_fail = false;
    check(a.reserve(11) == cudaSuccess && a && a.size() == 11, "a reserve after a failure allocates");

    void* const moved = a.get();
    A b(std::move(a));
    check(!a && a.size() == 0 && b.get() == moved && b.size() == 11, "the move constructor takes the allocation");
    {
      A c;
      check(c.reserve(5) == cudaSuccess && g_live.size() == 2, "a second allocation");
      c = std::move(b);
      check(!b && b.size() == 0 && c.get() == moved && c.size() == 11 && g_live.size() == 1,
            "move assignment frees the old allocation and takes the new");
      A d(std::move(c));
      check(g_live.size() == 1, "moving frees nothing");
    }
    check(g_live.empty(), "the last owner frees the allocation");
  }
  check(g_live.empty() && g_bad_frees == 0, "moved-from handles free nothing");
}

}  // namespace

extern "C" {
cudaError_t __wrap_cudaMalloc(void** p, size_t) { return fake_alloc(p); }
cudaError_t __wrap_cudaMallocHost(void** p, size_t) { return fake_alloc(p); }
cudaError_t __wrap_cudaFree(void* p) { return fake_free(p); }
cudaError_t __wrap_cudaFreeHost(void* p) { return fake_free(p); }
}

int main() {
  check_array<DeviceArray<double>>();
  check_array<PinnedArray<unsigned char>>();

  // without a device creation fails and leaves the handle empty; with one, the handle holds what was created
  Stream s;
  check((s.create() == cudaSuccess) == (static_cast<cudaStream_t>(s) != nullptr), "a stream holds what was created");
  Stream s2(std::move(s));
  check(static_cast<cudaStream_t>(s) == nullptr, "a moved-from stream is empty");
  Event e;
  check((e.create(cudaEventDisableTiming) == cudaSuccess) == (static_cast<cudaEvent_t>(e) != nullptr),
        "an event holds what was created");
  Event e2(std::move(e));
  check(static_cast<cudaEvent_t>(e) == nullptr, "a moved-from event is empty");
  std::printf("ok\n");
  return 0;
}
