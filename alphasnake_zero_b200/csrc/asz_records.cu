// asz_records.cu -- device-resident training records: the (root state, root Q) pairs Agent.make_moves appends when
// training (code/utils/agent.py:93-97) and the sampling + mirror augmentation of the trainer
// (code/utils/alpha_snake_zero_trainer.py:62-77, 93-100).
//
// The reference keeps two Python lists (Agent.records: (2H-1, 2W-1, 3) float32 arrays, Agent.values: float32[3]) and
// copies every root state to the host every root turn.  Here the planes of the root states are encoded by the fused
// tic/encode kernel straight into an engine-owned store in HBM (row_base = number of records so far), the root Q rows of
// the search are gathered next to them, and a training batch is one gather kernel that also writes the mirrored copy:
//   mirror_states = flip(states, axis=2)  (the width axis of [n, h, w, 3])      alpha_snake_zero_trainer.py:93-97
//   mirror_values = flip(values, axis=1)  (left <-> right)                       alpha_snake_zero_trainer.py:99-100
// Roofline: HBM bandwidth; algorithmic bytes per sampled record = plane read + 2 plane writes = 3 x 5,292 B at 11x11.
// Stored planes are asz_plane_pitch() floats apart (as the encode writes them); batches are dense.
#include <algorithm>
#include <cstdio>
#include <cstring>

#include "asz_engine.hpp"

namespace asz {

struct RecordStore {
  int64_t capacity = 0;      // rows
  int64_t count = 0;         // rows appended so far (host copy; refreshed by the synchronisation in asz_records_append)
  float* planes = nullptr;   // [capacity][pitch]: rows start on 32-byte sectors (asz_plane_pitch)
  float* values = nullptr;   // [capacity][3]
  int32_t* ids = nullptr;    // [capacity] game*8 + snake of every record
  int32_t* turns = nullptr;  // [capacity] append call (root turn) that produced the record
  int32_t n_appends = 0;
};

// values[base + i] = root_q[ids[base + i]] for the rows of the last encode launch
__global__ void records_values_kernel(const float* __restrict__ root_q, const int32_t* __restrict__ ids, const int32_t* __restrict__ n_rows,
                                      int64_t base, int64_t capacity, int32_t turn, float* __restrict__ values, int32_t* __restrict__ turns) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)*n_rows || base + i >= capacity) return;
  const int32_t id = ids[base + i];
  values[3 * (base + i)] = root_q[3 * (size_t)id];
  values[3 * (base + i) + 1] = root_q[3 * (size_t)id + 1];
  values[3 * (base + i) + 2] = root_q[3 * (size_t)id + 2];
  turns[base + i] = turn;
}

// One CTA per sampled record: X[i] = planes[idx[i]], V[i] = values[idx[i]]; when mirror: X[n + i] = flip(X[i], width axis),
// V[n + i] = reversed V[i].  A plane row is N pixels x 3 floats; the flipped row is the same pixels in reverse order.
__global__ void __launch_bounds__(256) records_gather_kernel(const float* __restrict__ planes, const float* __restrict__ values,
                                                             const int64_t* __restrict__ idx, int n, int N, int pitch, int mirror,
                                                             int64_t count, float* __restrict__ X, float* __restrict__ V) {
  const int i = (int)blockIdx.x;
  if (i >= n) return;
  const int64_t r = idx[i];
  const int plane = N * N * 3;
  float* x0 = X + (size_t)i * plane;
  float* x1 = X + (size_t)(n + i) * plane;
  if (r < 0 || r >= count) {            // out-of-range index: an all-NaN record (planes and values) is easier to notice than a silent zero
    const float nan = __int_as_float(0x7fc00000);
    for (int e = (int)threadIdx.x; e < plane; e += (int)blockDim.x) { x0[e] = nan; if (mirror) x1[e] = nan; }
    if (threadIdx.x < 3) {
      V[3 * (size_t)i + threadIdx.x] = nan;
      if (mirror) V[3 * (size_t)(n + i) + threadIdx.x] = nan;
    }
    return;
  }
  const float* src = planes + (size_t)r * pitch;
  for (int e = (int)threadIdx.x; e < plane; e += (int)blockDim.x) {
    const float v = src[e];
    x0[e] = v;
    if (mirror) {
      const int pix = e / 3, c = e - 3 * pix;
      const int y = pix / N, x = pix - y * N;
      x1[(y * N + (N - 1 - x)) * 3 + c] = v;
    }
  }
  if (threadIdx.x < 3) {
    const float v = values[3 * (size_t)r + threadIdx.x];
    V[3 * (size_t)i + threadIdx.x] = v;
    if (mirror) V[3 * (size_t)(n + i) + (2 - threadIdx.x)] = v;
  }
}

// the store grows (x2) when the next append might not fit: nothing is ever dropped because of a capacity guess
static int records_reserve(asz_engine* e, int64_t need_rows, cudaStream_t st) {
  RecordStore* r = e->records;
  if (need_rows <= r->capacity) return ASZ_OK;
  int64_t cap = r->capacity;
  while (cap < need_rows) cap *= 2;
  if (cap > 0x7fffffff) cap = 0x7fffffff;
  if (cap < need_rows) { set_error("record store cannot grow past 2^31 - 1 rows"); return ASZ_ERR_CAPACITY; }
  float *pl = nullptr, *va = nullptr; int32_t *ids = nullptr, *tu = nullptr;
  ASZ_CUDA(cudaMalloc(&pl, (size_t)cap * e->pitch * sizeof(float) + 32));
  ASZ_CUDA(cudaMalloc(&va, (size_t)cap * 3 * sizeof(float)));
  ASZ_CUDA(cudaMalloc(&ids, (size_t)cap * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&tu, (size_t)cap * sizeof(int32_t)));
  const size_t n = (size_t)r->count;
  ASZ_CUDA(cudaMemcpyAsync(pl, r->planes, n * e->pitch * sizeof(float), cudaMemcpyDeviceToDevice, st));
  ASZ_CUDA(cudaMemcpyAsync(va, r->values, n * 3 * sizeof(float), cudaMemcpyDeviceToDevice, st));
  ASZ_CUDA(cudaMemcpyAsync(ids, r->ids, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  ASZ_CUDA(cudaMemcpyAsync(tu, r->turns, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  ASZ_CUDA(cudaStreamSynchronize(st));
  cudaFree(r->planes); cudaFree(r->values); cudaFree(r->ids); cudaFree(r->turns);
  r->planes = pl; r->values = va; r->ids = ids; r->turns = tu; r->capacity = cap;
  return ASZ_OK;
}

void records_destroy(asz_engine* e) {
  RecordStore* r = e->records;
  if (!r) return;
  cudaFree(r->planes); cudaFree(r->values); cudaFree(r->ids); cudaFree(r->turns);
  delete r;
  e->records = nullptr;
}

}  // namespace asz

using namespace asz;

extern "C" {

int asz_records_enable(asz_engine* e, int64_t capacity_rows) {
  if (!e || capacity_rows < 1) { set_error("asz_records_enable: bad argument"); return ASZ_ERR_ARG; }
  if (capacity_rows > 0x7fffffff) { set_error("asz_records_enable: capacity must fit 31 bits"); return ASZ_ERR_ARG; }
  DeviceGuard guard(e->device);
  records_destroy(e);
  RecordStore* r = new RecordStore();
  e->records = r;
  r->capacity = capacity_rows;
  ASZ_CUDA(cudaMalloc(&r->planes, (size_t)capacity_rows * e->pitch * sizeof(float) + 32));
  ASZ_CUDA(cudaMalloc(&r->values, (size_t)capacity_rows * 3 * sizeof(float)));
  ASZ_CUDA(cudaMalloc(&r->ids, (size_t)capacity_rows * sizeof(int32_t)));
  ASZ_CUDA(cudaMalloc(&r->turns, (size_t)capacity_rows * sizeof(int32_t)));
  return ASZ_OK;
}

// agent.py:93-97 for every live snake of every live root game: the current root state and the root Q row of the search
// that just finished (asz_search_finish).  d_root_q: [games*8][3] or NULL = the engine's own buffer.  Synchronises the
// stream (the number of records is needed on the host); *h_count = records held afterwards.
int asz_records_append(asz_engine* e, const float* d_root_q, int64_t* h_count, void* stream) {
  if (!e || !e->records) { set_error("asz_records_append: records are not enabled"); return ASZ_ERR_STATE; }
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:records append");
  RecordStore* r = e->records;
  cudaStream_t st = (cudaStream_t)stream;
  const float* q = d_root_q ? d_root_q : asz_search_root_q(e);
  if (!q) { set_error("asz_records_append: no root Q (search not configured and d_root_q is null)"); return ASZ_ERR_STATE; }
  int rc = records_reserve(e, r->count + (int64_t)e->cfg.games * e->cfg.snakes, st);
  if (rc != ASZ_OK) return rc;
  asz_step_args a;
  memset(&a, 0, sizeof a);
  a.flags = ASZ_STEP_ENCODE; a.spawn_mode = ASZ_SPAWN_NONE;
  a.d_planes = r->planes; a.d_row_ids = r->ids; a.max_rows = (int32_t)r->capacity; a.row_base = (int32_t)r->count;
  a.plane_pitch = e->pitch;
  a.d_row_count = e->rows_ptr();
  rc = asz_env_step(e, &a, stream);
  if (rc != ASZ_OK) return rc;
  const int64_t room = r->capacity - r->count;
  const int64_t max_new = std::min<int64_t>(room, (int64_t)e->cfg.games * e->cfg.snakes);
  if (max_new > 0) {
    records_values_kernel<<<(unsigned)((max_new + 255) / 256), 256, 0, st>>>(q, r->ids, e->rows_ptr(), r->count, r->capacity, r->n_appends,
                                                                            r->values, r->turns);
    if (!cuda_ok(cudaGetLastError(), "records_values_kernel")) return ASZ_ERR_CUDA;
  }
  int32_t rows = 0;
  ASZ_CUDA(cudaMemcpyAsync(&rows, e->rows_ptr(), sizeof rows, cudaMemcpyDeviceToHost, st));
  ASZ_CUDA(cudaStreamSynchronize(st));
  r->n_appends += 1;
  if ((int64_t)rows > room) {
    r->count = r->capacity;
    if (h_count) *h_count = r->count;
    char msg[160];
    snprintf(msg, sizeof msg, "record store full: %d new records, room for %lld of %lld (raise the capacity of asz_records_enable)",
             rows, (long long)room, (long long)r->capacity);
    set_error(msg);
    return ASZ_ERR_CAPACITY;
  }
  r->count += rows;
  if (h_count) *h_count = r->count;
  return ASZ_OK;
}

int asz_records_count(asz_engine* e, int64_t* h_count) {
  if (!e || !e->records || !h_count) { set_error("records are not enabled"); return ASZ_ERR_STATE; }
  *h_count = e->records->count;
  return ASZ_OK;
}

// Agent.clear (agent.py:140-147) for the records
int asz_records_clear(asz_engine* e) {
  if (!e || !e->records) { set_error("records are not enabled"); return ASZ_ERR_STATE; }
  e->records->count = 0;
  e->records->n_appends = 0;
  return ASZ_OK;
}

// alpha_snake_zero_trainer.py:70-77: X = [records[i] for i in indexs], V likewise, then X += mirror_states(X), V += mirror_values(V).
// d_idx: [n] int64 record indices (the reference draws them on the host with random.sample).  d_X: [(mirror ? 2 : 1) * n][plane]
// float32, d_V: [(mirror ? 2 : 1) * n][3]; the mirrored copies follow the n originals, in the same order.
int asz_records_gather(asz_engine* e, const int64_t* d_idx, int32_t n, int32_t mirror, float* d_X, float* d_V, void* stream) {
  if (!e || !e->records) { set_error("records are not enabled"); return ASZ_ERR_STATE; }
  if (!d_idx || !d_X || !d_V || n < 0) { set_error("asz_records_gather: bad argument"); return ASZ_ERR_ARG; }
  if (n == 0) return ASZ_OK;
  DeviceGuard guard(e->device);
  NvtxRange nvtx("asz:records gather + mirror");
  RecordStore* r = e->records;
  records_gather_kernel<<<n, 256, 0, (cudaStream_t)stream>>>(r->planes, r->values, d_idx, n, 2 * e->cfg.side - 1, e->pitch, mirror ? 1 : 0, r->count,
                                                            d_X, d_V);
  return cuda_ok(cudaGetLastError(), "records_gather_kernel") ? ASZ_OK : ASZ_ERR_CUDA;
}

float* asz_records_planes(asz_engine* e) { return (e && e->records) ? e->records->planes : nullptr; }
float* asz_records_values(asz_engine* e) { return (e && e->records) ? e->records->values : nullptr; }
int32_t* asz_records_ids(asz_engine* e) { return (e && e->records) ? e->records->ids : nullptr; }
int32_t* asz_records_turns(asz_engine* e) { return (e && e->records) ? e->records->turns : nullptr; }

}  // extern "C"
