// DirectSession for one B200 graph copy.
//
// BASELINE.json keeps the reference's DirectSession/executor "as-is"; those sources cannot be
// compiled here (no bazel/protoc/Eigen), so this class reproduces the CALL CONTRACT the kernels
// see from them and nothing more:
//   * Run() prunes the graph to the fetches/targets, stopping at feeds
//     (direct_session.cc:1098-1233), caches the result under a feeds/fetches/targets key
//     (GetOrCreateExecutors :904-1096) and creates each kernel once with CreateOpKernel
//     (:1028-1042; stateful kernels such as VariableV2 therefore keep their state);
//   * the executor walks the partition in a topological order on ONE host thread -- what
//     ExecutorState::Process does for a GPU partition, whose kernels are all "inexpensive"
//     (executor.cc:1487-1691, op_kernel.cc:97-99) -- filling OpKernelContext::Params
//     (:1575-1649), calling Device::Compute (:1651) and propagating outputs (:1654-1673);
//   * kernels whose op is a collective (B200AllReduce*) are placed on the device's collective
//     stream when replicas > 1 (the reference's per-node DeviceContext / stream assignment,
//     gpu_device.cc:337-399, executor.cc:1575-1649): the executor orders the two streams with
//     events, keeps every tensor such a node touched alive until the step's sync, and schedules
//     collectives as soon as their inputs exist so they overlap the rest of the backward pass;
//   * feeds are copied host->device and fetches device->host through the device context
//     (the job of _Send/_Recv + GPUUtil), and the device is synced exactly once per step
//     (sync_on_finish, direct_session.cc:451, executor.cc:2211-2217).
// Everything is placed on DEVICE_GPU: the named ops have no CPU fallback by design.
#ifndef B200TF_CORE_COMMON_RUNTIME_DIRECT_SESSION_H_
#define B200TF_CORE_COMMON_RUNTIME_DIRECT_SESSION_H_

#include <chrono>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "tensorflow/core/common_runtime/gpu/gpu_device.h"
#include "tensorflow/core/framework/op_kernel.h"
#include "tensorflow/core/public/session.h"

namespace tensorflow {

class DirectSession : public Session {
 public:
  explicit DirectSession(const SessionOptions& options);
  ~DirectSession() override;
  Status Init();
  Status Create(const GraphDef& graph) override;
  Status Extend(const GraphDef& graph) override;
  Status Run(const std::vector<std::pair<std::string, Tensor>>& inputs,
             const std::vector<std::string>& output_tensor_names,
             const std::vector<std::string>& target_node_names,
             std::vector<Tensor>* outputs) override;
  Status Close() override;
  const RunStats& last_run_stats() const override { return stats_; }
  Status StageFeed(const Tensor& host, Tensor* staged) override;
  BaseGPUDevice* device() const { return device_.get(); }

 private:
  struct TensorId {
    int node = -1;
    int slot = 0;
  };
  struct NodeItem {
    NodeDef def;
    std::vector<TensorId> inputs;       // data inputs, in op-signature order
    std::vector<int> control_inputs;    // node indices
    std::unique_ptr<OpKernel> kernel;   // created on first use
    std::string unsupported;            // non-empty: op type not registered (imported graphs)
  };
  struct InputSource {
    int feed = -1;  // >= 0: index into the step's feeds
    TensorId id;    // otherwise: produced by this (node, slot)
  };
  struct PlanNode {
    int node;            // index into nodes_ (-1 for a node synthesised by a rewrite)
    NodeItem* item;      // the node to execute (owned by nodes_ or by ExecutorsAndKeys::rewritten)
    bool dead = false;   // folded into a fused node by a rewrite
    int collective = -1; // >= 0: runs on the collective stream; index of its event pair
    int arena = -1;      // >= 0: a B200AllReduceN whose inputs are laid out in this gradient arena
    // per output: (arena, position) when the output is one of an arena's gradients, else (-1, -1)
    std::vector<std::pair<int, int>> arena_slots;
    std::vector<InputSource> inputs;
    int first_entry;  // index of output slot 0 in the entry table
    // A node synthesised from several graph nodes may deliver its outputs to entries that are
    // not consecutive (empty: output o lives in first_entry + o).
    std::vector<int> output_entries;
    int out_entry(int o) const {
      return output_entries.empty() ? first_entry + o : output_entries[o];
    }
  };
  // Gradient arena (the job of later TensorFlow's ScopedAllocator): the tensors one
  // B200AllReduceN reduces are produced directly into consecutive 256-byte-aligned windows of
  // one buffer, so the bucket is ONE in-place ncclAllReduce with no gather/scatter copies.
  // Sizes are learned from the first step that runs the plan; a producer whose request does not
  // match its window simply allocates normally and the collective falls back to its copying path.
  struct GradientArena {
    std::vector<size_t> bytes, offsets;
    size_t total = 0;
    DataType dtype = DT_FLOAT;
    bool learned = false;
  };
  struct ExecutorsAndKeys {
    std::vector<PlanNode> order;
    std::vector<GradientArena> arenas;
    std::vector<std::unique_ptr<NodeItem>> rewritten;  // fused nodes created for this plan
    std::vector<InputSource> fetches;
    std::vector<int> node_first_entry;  // per graph node: entry index of its output 0 (-1: pruned)
    std::vector<int> entry_consumers;   // per entry: how many plan inputs read it
    std::vector<bool> entry_is_fetch;
    std::vector<bool> feed_needs_device, feed_needs_host;
    int num_entries = 0;
    // per collective-stream node: [2k] inputs-ready (recorded on compute), [2k+1] done
    std::vector<std::unique_ptr<gpu::Event>> collective_events;
    // ---- step-level CUDA graph of this plan (the executor cache entry of
    // direct_session.cc:918-936 holding its whole launch sequence).  Eligible plans (no feeds, one
    // stream, no host round trips) are captured on their third run and replayed afterwards.
    struct CapturedFetch {
      Tensor value;             // a plain value: the tensor the captured kernels write
      Tensor* ref = nullptr;    // a variable: read at fetch time (its buffer is stable)
      std::mutex* ref_mu = nullptr;
      bool on_host = false;
    };
    int graph_state = 0;        // 0 unknown, 1 eligible (counting warm runs), 2 captured, -1 never
    int warm_runs = 0;
    void* graph_exec = nullptr;
    long long graph_launches = 0;             // kernels per replay (for the launch counter)
    unsigned long long graph_peer_collectives = 0, graph_nccl_collectives = 0;
    std::vector<void*> graph_pinned;          // device memory the captured kernels address
    std::vector<Tensor> graph_keepalive;      // entries alive at the end of the captured walk
    std::vector<CapturedFetch> graph_fetches;
    bool has_assign = false;                  // running this plan may move a variable's buffer
  };
  struct Entry {
    Tensor val;
    Tensor* ref = nullptr;
    std::mutex* ref_mu = nullptr;
    bool has_value = false;
    bool on_host = false;
    gpu::Event* pending = nullptr;  // produced on another stream: wait for this before reading
  };
  struct StagedFeed {
    std::unique_ptr<gpu::Event> ready;
    Tensor host;  // keeps the pinned source alive until the copy has been consumed
  };

  static int entry_index_of(const ExecutorsAndKeys* ek, const TensorId& id) {
    return ek->node_first_entry[id.node] + id.slot;
  }
  static Status ParseTensorName(const std::string& name, std::string* node, int* slot);
  Status AddNodes(const GraphDef& graph);
  Status AddNodesImpl(const GraphDef& graph);
  Status GetOrCreateExecutors(const std::vector<std::string>& feeds,
                              const std::vector<std::string>& fetches,
                              const std::vector<std::string>& targets, ExecutorsAndKeys** out);
  Status EnsureKernel(NodeItem* item);
  // GraphOptimizer-stage rewrite (direct_session.cc:1051 role): MatMul+BiasAdd(+Relu) and
  // MatMul+ReluGrad chains whose intermediates have a single consumer run as one _FusedMatMul.
  Status FuseMatMulChains(ExecutorsAndKeys* ek);
  // A dense layer's dX and dW products (two MatMuls reading the same tensor, neither depending on
  // the other) run as one _MatMulPair: one persistent GEMM launch for both.
  Status FuseSiblingMatMuls(ExecutorsAndKeys* ek);
  // SoftmaxCrossEntropyWithLogits whose backprop output only feeds Mul(backprop, scalar Const)
  // (the gradient of a mean loss, nn_grad.py:323-333 + math_grad.py _MeanGrad) runs as one
  // _ScaledSoftmaxCrossEntropyWithLogits: same fp32 roundings, one pass less over [batch, classes].
  Status FuseXentScale(ExecutorsAndKeys* ek);
  // Runs of ApplyGradientDescent nodes separated only by Const nodes (what an optimizer emits)
  // become one _MultiApplyGradientDescent: one launch instead of one per variable.
  Status FuseApplyGradientDescent(ExecutorsAndKeys* ek);
  // CUDA-graph capture / replay of a whole step (direct_session.cc, "step-level CUDA graphs")
  bool GraphEligible(ExecutorsAndKeys* ek, size_t num_feeds);
  Status ReplayGraph(ExecutorsAndKeys* ek, std::vector<Tensor>* outputs);
  void DropGraph(ExecutorsAndKeys* ek);
  void DropAllGraphs();
  Status FuseReluGradBiasGrad(ExecutorsAndKeys* ek);
  Status FusePoolGradReluGradBiasGrad(ExecutorsAndKeys* ek);
  Status MergeAllReduceBuckets(ExecutorsAndKeys* ek);
  void PlanGradientArenas(ExecutorsAndKeys* ek);
  Status RunPlan(ExecutorsAndKeys* ek, const std::vector<std::pair<std::string, Tensor>>& inputs,
                 std::vector<Tensor>* outputs);

  const SessionOptions options_;
  std::unique_ptr<BaseGPUDevice> device_;
  std::mutex mu_;
  std::vector<std::unique_ptr<NodeItem>> nodes_;
  std::unordered_map<std::string, int> node_index_;
  std::map<std::string, std::unique_ptr<ExecutorsAndKeys>> executors_;
  RunStats stats_;
  std::unordered_map<const TensorBuffer*, StagedFeed> staged_;  // copies still in flight
  std::chrono::steady_clock::time_point run_start_;
  long long step_id_ = 0;
  bool closed_ = false;
};

}  // namespace tensorflow
#endif
