// Internal plan structure shared by engine.cu and conv_tc.cu (not part of the C ABI).
#pragma once
#include <map>
#include <string>

#include "common.cuh"

namespace lstur {
struct Region {
  size_t off;       // bytes into workspace (ws) / floats into the dense arena (dense)
  long long count;  // elements (4-byte)
};
}  // namespace lstur

struct lstur_plan {
  lstur_config c;
  int N, Nh, Nc, Lp, D;
  std::map<std::string, lstur::Region> ws;     // workspace regions
  std::map<std::string, lstur::Region> dense;  // dense-parameter layout (off in floats)
  size_t ws_bytes = 0;
  long long dense_count = 0;
  size_t gemm_ws_bytes = 0;
  bool tc_gru = false;      // the GRU recurrence runs on tcgen05 (gru_tc.cu): tensor-core precision, lstur_gru_tc_supported
  // optional CUDA events recorded around one kernel of the step (bench.py roofline probe)
  int probe_id = 0;
  cudaEvent_t probe_start = nullptr, probe_stop = nullptr;
  // the 16-bit copy of the (frozen) word table in the workspace is re-packed only when its source / destination
  // changes or lstur_plan_invalidate_tables() was called (the table was written)
  const void* emb16_src = nullptr;
  void* emb16_dst = nullptr;
  // data-parallel overlap: recorded by lstur_backward once every gradient except the title-encoder bucket (conv_w, conv_b,
  // att_w, att_b = the first dense_head floats of the arena) and the user-row gradients are final
  cudaEvent_t ev_tail_ready = nullptr;
  long long dense_head = 0;
  unsigned last_seed = 0;   // seed / mode of the last forward (backward replays its dropout streams)
  int last_training = 0;
  int last_aux = 0;        // the last forward ran the auxiliary vertical classifier (labels were given)
  int last_cls_n = 0;      // titles of the last lstur_title_cls_forward
};

namespace lstur {
template <typename T>
inline T* W(const lstur_plan* p, void* ws, const char* name) {
  auto it = p->ws.find(name);
  return it == p->ws.end() ? nullptr : (T*)((char*)ws + it->second.off);
}
inline const float* DP(const lstur_plan* p, const float* dense, const char* name) {
  auto it = p->dense.find(name);
  return it == p->dense.end() ? nullptr : dense + it->second.off;
}
inline float* DG(const lstur_plan* p, float* dense, const char* name) {
  auto it = p->dense.find(name);
  return it == p->dense.end() ? nullptr : dense + it->second.off;
}
}  // namespace lstur

#define PROBE_BEGIN(p, id, st) do { if ((p)->probe_id == (id) && (p)->probe_start) cudaEventRecord((p)->probe_start, st); } while (0)
#define PROBE_END(p, id, st) do { if ((p)->probe_id == (id) && (p)->probe_stop) cudaEventRecord((p)->probe_stop, st); } while (0)

#define RC(x)              \
  do {                     \
    int rc__ = (x);        \
    if (rc__) return rc__; \
  } while (0)
