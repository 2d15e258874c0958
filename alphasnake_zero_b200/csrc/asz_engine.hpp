// asz_engine.hpp -- host-side engine object behind the C ABI (include/asz_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>

#include <string>

#include "../../include/asz_b200.h"

namespace asz {

void set_error(const std::string& msg);
bool cuda_ok(cudaError_t err, const char* what);

#define ASZ_CUDA(call)                                         \
  do {                                                         \
    if (!::asz::cuda_ok((call), #call)) return ASZ_ERR_CUDA;   \
  } while (0)

struct SearchState;   // asz_mcts.cu
struct RecordStore;   // asz_records.cu
struct PitState;      // asz_pit.cu

// Every entry point that takes an engine (or a network) runs on THAT object's device, whatever device is current in the
// calling thread ("one engine per GPU": several engines on different GPUs may live in one process).
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    int cur = -1;
    if (cudaGetDevice(&cur) == cudaSuccess && cur != dev && cudaSetDevice(dev) == cudaSuccess) prev = cur;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};
// NVTX range per phase (tic / encode, probe, net, sample, finish, records): visible in Nsight Systems / ncu --nvtx, a
// no-op function-pointer check when no tool is attached (SURVEY.md section 5, tracing row)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};
constexpr int kMaxDevices = 64;   // per-device "kernel attributes configured" flags (function attributes are per device)
constexpr size_t kSchedBytes = 128;   // asz_engine::row_count: the env kernel's two alternating scheduling words, 64 bytes apart

// Device-resident game set: one record per game, structure-of-arrays over games.
//   cells  [n][PC]  u16 stamps (asz_common.cuh)
//   snakes [n][8]   u64 packed snake records
//   meta   [n][8]   u32 turn, episode, wall, body, head, starve, food_eaten, flags
struct GameSet {
  int n = 0;
  uint16_t* cells = nullptr;
  uint64_t* snakes = nullptr;
  uint32_t* meta = nullptr;
};

}  // namespace asz

struct asz_engine {
  asz_config cfg;
  int device = 0;
  int n_sm = 0;          // multiprocessors of `device`
  int pc = 0;            // padded cells per game
  int plane = 0;         // floats per plane
  int pitch = 0;         // floats between consecutive planes of the engine's own buffers (plane rounded up to 8: 32-byte rows)
  uint32_t chance_thresh = 0;
  asz::GameSet root;
  // env-step scratch owned by the engine
  float* planes = nullptr;        // [G*S][pitch]
  int32_t* row_ids = nullptr;     // [G*S]
  int32_t* row_count = nullptr;   // kSchedBytes: the kernel's 64-bit scheduling words (rows handed out | tickets handed out)
  int sched_flip = 0;             // launches alternate between the word at byte 0 and the one at byte 64 (asz_env_step)
  // the word of the LAST launch: its low half is that launch's row count
  int32_t* rows_ptr() const { return reinterpret_cast<int32_t*>(reinterpret_cast<char*>(row_count) + (sched_flip ? 64 : 0)); }
  unsigned long long* totals = nullptr;  // [32]: [0..15] totals (asz_get_totals), [16..23] the profile build's cycle sums
  // asz_env_submit_host / asz_env_wait_host: two steps in flight, the inputs of the next one copied under the kernel of this one
  struct HostPipe {
    bool ready = false;
    cudaStream_t copy = nullptr;                 // host -> device copies of the steps' inputs
    cudaStream_t copy_out = nullptr;             // device -> host copies of the steps' results
    cudaEvent_t copied[2] = {nullptr, nullptr};  // slot's inputs are on the device
    cudaEvent_t stepped[2] = {nullptr, nullptr}; // slot's launch has finished
    cudaEvent_t done[2] = {nullptr, nullptr};    // slot's launch and result copies have finished
    uint8_t* actions[2] = {nullptr, nullptr};    // [G*8] per slot
    int32_t* spawn[2] = {nullptr, nullptr};      // [G] per slot
    uint8_t* d_ended[2] = {nullptr, nullptr};    // [G] per slot: the kernel's per-game results before they travel
    int8_t* d_rewards[2] = {nullptr, nullptr};   // [G*8] per slot
    int32_t* d_rows[2] = {nullptr, nullptr};     // the step's row count
    int32_t* h_rows = nullptr;                   // pinned, one 64-byte line per slot
    bool busy[2] = {false, false};
    int next = 0;
  } hostpipe;
  asz::SearchState* search = nullptr;
  asz::RecordStore* records = nullptr;   // device-resident training records (asz_records_*)
  asz::PitState* pit = nullptr;          // two-network match (asz_pit_*), allocated by the first asz_pit_begin
  asz_engine* pit_searcher[2] = {nullptr, nullptr};   // asz_pit_set_search: the search engine of Alice / Bob, not owned
};

namespace asz {
int gameset_alloc(GameSet& gs, int n, int pc);
void gameset_free(GameSet& gs);
int search_create(asz_engine* e);
void search_destroy(asz_engine* e);
// stand-in value function of asz_search_stub_values: which word of the plane key it reads (1 unless a pit side says otherwise)
void search_set_stub_word(asz_engine* e, int word);
void records_destroy(asz_engine* e);
void pit_destroy(asz_engine* e);
void host_pipe_destroy(asz_engine* e);
// board side and device of a value network (asz_net.cu)
int net_side(const asz_net* n);
int net_device(const asz_net* n);
}  // namespace asz
