// loop_graph.cuh -- the CUDA graphs of the device-side loops (evaluate.cu, selfplay.cu): one graph per workspace, whose single WHILE
// conditional node repeats a captured body until a kernel of the body writes 0 into the node's handle.  A graph is built on the first
// call for a workspace, kept with it (like the auxiliary streams of EAZ_FLAG_STREAMS) and rebuilt when anything it bakes in changes;
// each caller describes what its body bakes in by its own record type.
#pragma once
#include <cstring>
#include <mutex>
#include <string>

#include "common.cuh"

namespace eaz {

inline bool same_env(const eaz_env& a, const eaz_env& b) {
  return a.kind == b.kind && a.size == b.size && a.action_map == b.action_map && a.word_size == b.word_size &&
         a.binary_encoding == b.binary_encoding && a.reward_fn == b.reward_fn;
}
inline bool same_net(const eaz_fc_params& a, const eaz_fc_params& b) {
  return a.in_dim == b.in_dim && a.hidden == b.hidden && a.num_actions == b.num_actions && !memcmp(a.w, b.w, sizeof(a.w)) &&
         !memcmp(a.b, b.b, sizeof(a.b)) && a.binary_set == b.binary_set && a.hash_bits == b.hash_bits && a.hash_io == b.hash_io &&
         a.word_size == b.word_size && !memcmp(&a.max_u, &b.max_u, sizeof(float)) && !memcmp(&a.novelty_scale, &b.novelty_scale, sizeof(float));
}

// Captures body(capture_stream, handle) into a WHILE node whose handle starts at 1 (the loop always runs its first iteration) and
// instantiates the graph; on success *graph / *exec hold the new graph (the old ones are destroyed).
template <typename Body>
int build_loop_graph(const char* what, cudaStream_t* capture, cudaGraph_t* graph_io, cudaGraphExec_t* exec_io, Body&& body) {
  const std::string w(what);
  if (!*capture)
    if (cudaError_t e = cudaStreamCreateWithFlags(capture, cudaStreamNonBlocking); e != cudaSuccess) return cuda_fail(e, (w + " capture stream").c_str());
  cudaGraph_t graph = nullptr;
  if (cudaError_t e = cudaGraphCreate(&graph, 0); e != cudaSuccess) return cuda_fail(e, (w + " graph").c_str());
  auto fail = [&](cudaError_t e, const char* part) {
    cudaGraphDestroy(graph);
    return cuda_fail(e, (w + part).c_str());
  };
  cudaGraphConditionalHandle handle;
  if (cudaError_t e = cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault); e != cudaSuccess)
    return fail(e, " conditional handle");
  cudaGraphNodeParams p{};
  p.type = cudaGraphNodeTypeConditional;
  p.conditional.handle = handle;
  p.conditional.type = cudaGraphCondTypeWhile;
  p.conditional.size = 1;
  cudaGraphNode_t node;
  if (cudaError_t e = cudaGraphAddNode(&node, graph, nullptr, 0, &p); e != cudaSuccess) return fail(e, " WHILE node");
  cudaGraph_t body_graph = p.conditional.phGraph_out[0];
  if (cudaError_t e = cudaStreamBeginCaptureToGraph(*capture, body_graph, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed); e != cudaSuccess)
    return fail(e, " body capture");
  const int rc = body(*capture, handle);
  cudaGraph_t captured = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(*capture, &captured);  // (always: the stream must leave capture mode)
  if (rc) {
    cudaGraphDestroy(graph);
    return rc;
  }
  if (ce != cudaSuccess) return fail(ce, " body capture");
  cudaGraphExec_t exec = nullptr;
  if (cudaError_t e = cudaGraphInstantiate(&exec, graph, 0); e != cudaSuccess) return fail(e, " graph instantiate");
  if (*exec_io) cudaGraphExecDestroy(*exec_io);  // (an in-flight launch of the old one completes first)
  if (*graph_io) cudaGraphDestroy(*graph_io);
  *graph_io = graph;
  *exec_io = exec;
  return 0;
}

// The graphs of one kind of loop, one per (workspace, device).  Rec: what the body bakes in, with `bool same(const Rec&) const`.
template <typename Rec, int kSlots = 64>
struct LoopGraphs {
  struct Slot {
    bool used = false;
    int device = -1;
    const void* workspace = nullptr;
    Rec rec;
    cudaStream_t capture = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
  };
  Slot slots[kSlots];
  std::mutex mu;  // the caller holds it for the whole enqueue of one call

  Slot* slot(const void* workspace, int dev) {
    for (auto& g : slots)
      if (g.used && g.workspace == workspace && g.device == dev) return &g;
    for (auto& g : slots)
      if (!g.used) return &g;
    // table full: reuse a slot of this device (its graph is rebuilt for this workspace)
    const size_t h = ((uintptr_t)workspace >> 8) * 0x9E3779B97F4A7C15ull >> 32;
    for (int k = 0; k < kSlots; ++k) {
      Slot* g = &slots[(h + k) % kSlots];
      if (g->device == dev) return g;
    }
    return nullptr;
  }

  // Launches the graph of `workspace` on `st`, (re)built first unless it exists and bakes in `rec`.
  template <typename Body>
  int launch(const char* what, const void* workspace, const Rec& rec, cudaStream_t st, Body&& body) {
    cudaGraphExec_t exec = nullptr;
    if (int rc = build(what, workspace, rec, &exec, body)) return rc;
    if (cudaError_t e = cudaGraphLaunch(exec, st); e != cudaSuccess) return cuda_fail(e, (std::string(what) + " graph launch").c_str());
    return 0;
  }

  // The graph of `workspace` in *exec, (re)built unless it exists and bakes in `rec`.
  template <typename Body>
  int build(const char* what, const void* workspace, const Rec& rec, cudaGraphExec_t* exec, Body&& body) {
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev); e != cudaSuccess) return cuda_fail(e, (std::string(what) + " device").c_str());
    Slot* g = slot(workspace, dev);
    if (!g) {
      set_error("%s: no graph slot for this device", what);
      return EAZ_ERR_CUDA;
    }
    if (!(g->used && g->workspace == workspace && g->device == dev && g->exec && g->rec.same(rec))) {
      g->used = true;  // (the slot is this workspace's from now on; a failed build leaves exec NULL and is retried next call)
      g->workspace = workspace;
      g->device = dev;
      if (g->exec) {
        cudaGraphExecDestroy(g->exec);
        g->exec = nullptr;
      }
      if (int rc = build_loop_graph(what, &g->capture, &g->graph, &g->exec, body)) return rc;
      g->rec = rec;
    }
    *exec = g->exec;
    return 0;
  }
};

}  // namespace eaz
