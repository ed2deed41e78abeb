#include "tensorflow/core/common_runtime/direct_session.h"

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <queue>
#include <set>

namespace tensorflow {

// Environment switch that defaults to ON: only an explicit "0" turns it off.
static bool EnvFlagOff(const char* name) {
  const char* v = getenv(name);
  return v != nullptr && std::strcmp(v, "0") == 0;
}

Status NewSession(const SessionOptions& options, Session** out_session) {
  if (!options.target.empty())
    return errors::Unimplemented("Only the in-process DirectSession (target \"\") is available; "
                                 "the gRPC runtime is outside the B200 hot path");
  std::unique_ptr<DirectSession> s(new DirectSession(options));
  TF_RETURN_IF_ERROR(s->Init());
  *out_session = s.release();
  return Status::OK();
}

DirectSession::DirectSession(const SessionOptions& options) : options_(options) {}

DirectSession::~DirectSession() {
  if (device_) device_->Sync();
  if (device_) DropAllGraphs();  // graphs and the memory they pin go before the plans
  executors_.clear();
  nodes_.clear();  // kernels (and the variables they own) go before the device's allocator
}

Status DirectSession::Init() {
  TF_RETURN_IF_ERROR(
      BaseGPUDevice::Create(options_.gpu_device_id, options_.gpu_memory_limit_bytes, &device_));
  device_->set_collective_comm(options_.collective_comm, options_.num_replicas);
  return Status::OK();
}

Status DirectSession::ParseTensorName(const std::string& name, std::string* node, int* slot) {
  const size_t colon = name.rfind(':');
  if (colon == std::string::npos) {
    *node = name;
    *slot = 0;
    return Status::OK();
  }
  *node = name.substr(0, colon);
  const std::string idx = name.substr(colon + 1);
  if (idx.empty() || idx.find_first_not_of("0123456789") != std::string::npos)
    return errors::InvalidArgument("Malformed tensor name '", name, "'");
  *slot = atoi(idx.c_str());
  return Status::OK();
}

Status DirectSession::AddNodes(const GraphDef& graph) {
  // Transactional, like the reference's Extend (a failed GraphDef leaves the session's graph
  // unchanged, direct_session.cc ExtendLocked): on any error roll nodes_ / node_index_ back.
  const size_t rollback_to = nodes_.size();
  Status s = AddNodesImpl(graph);
  if (!s.ok()) {
    for (size_t i = rollback_to; i < nodes_.size(); ++i) node_index_.erase(nodes_[i]->def.name);
    nodes_.resize(rollback_to);
  }
  return s;
}

Status DirectSession::AddNodesImpl(const GraphDef& graph) {
  const size_t first_new = nodes_.size();
  for (const NodeDef& nd : graph.node) {
    if (node_index_.count(nd.name))
      return errors::InvalidArgument("Node '", nd.name, "' is not unique");
    const OpDef* op_def = OpRegistry::Global()->LookUp(nd.op);
    std::unique_ptr<NodeItem> item(new NodeItem);
    item->def = nd;
    if (op_def == nullptr) {
      // Imported graphs (TF_GraphImportGraphDef) carry savers, string ops, parsers ... that this
      // runtime does not implement: such a node only fails a Run() that actually needs it.
      item->unsupported = strings::StrCat("Op type not registered '", nd.op, "' (node '", nd.name,
                                          "'): outside the B200 hot path");
      node_index_[nd.name] = static_cast<int>(nodes_.size());
      nodes_.push_back(std::move(item));
      continue;
    }
    TF_RETURN_IF_ERROR(ValidateNodeDef(&item->def, *op_def));
    // Explicit /cpu:0 placements (imported inference graphs pin their string / parsing front
    // end there) are accepted and ignored: every node this runtime can run runs on the GPU.
    node_index_[nd.name] = static_cast<int>(nodes_.size());
    nodes_.push_back(std::move(item));
  }
  // resolve inputs after all nodes of this batch are known (GraphDefs need not be sorted)
  for (size_t i = first_new; i < nodes_.size(); ++i) {
    NodeItem* item = nodes_[i].get();
    for (const std::string& in : item->def.input) {
      if (!in.empty() && in[0] == '^') {
        auto it = node_index_.find(in.substr(1));
        if (it == node_index_.end())
          return errors::InvalidArgument("Node '", item->def.name, "': Unknown control input '", in, "'");
        item->control_inputs.push_back(it->second);
        continue;
      }
      std::string src;
      int slot;
      TF_RETURN_IF_ERROR(ParseTensorName(in, &src, &slot));
      auto it = node_index_.find(src);
      if (it == node_index_.end())
        return errors::InvalidArgument("Node '", item->def.name, "': Unknown input node '", in, "'");
      item->inputs.push_back(TensorId{it->second, slot});
    }
    if (!item->unsupported.empty()) continue;
    const OpDef* op_def = OpRegistry::Global()->LookUp(item->def.op);
    DataTypeVector in_types, out_types;
    TF_RETURN_IF_ERROR(InOutTypesForNode(item->def, *op_def, &in_types, &out_types));
    if (in_types.size() != item->inputs.size())
      return errors::InvalidArgument("Node '", item->def.name, "' of type ", item->def.op,
                                     " expects ", in_types.size(), " inputs but has ",
                                     item->inputs.size());
  }
  return Status::OK();
}

Status DirectSession::Create(const GraphDef& graph) {
  std::lock_guard<std::mutex> l(mu_);
  if (!nodes_.empty())
    return errors::AlreadyExists("A Graph has already been created for this session.");
  return AddNodes(graph);
}

Status DirectSession::Extend(const GraphDef& graph) {
  std::lock_guard<std::mutex> l(mu_);
  if (closed_) return errors::Cancelled("Session has been closed.");
  return AddNodes(graph);
}

Status DirectSession::Close() {
  std::lock_guard<std::mutex> l(mu_);
  closed_ = true;
  if (device_) return device_->Sync();
  return Status::OK();
}

Status DirectSession::EnsureKernel(NodeItem* item) {
  if (item->kernel) return Status::OK();
  return CreateOpKernel(DeviceType(DEVICE_GPU), device_.get(),
                        device_->GetAllocator(AllocatorAttributes()), item->def, &item->kernel);
}

Status DirectSession::GetOrCreateExecutors(const std::vector<std::string>& feeds,
                                           const std::vector<std::string>& fetches,
                                           const std::vector<std::string>& targets,
                                           ExecutorsAndKeys** out) {
  // Same key construction idea as direct_session.cc:918-936 (sorted names joined).
  std::vector<std::string> fs(feeds), ts(targets);
  std::sort(ts.begin(), ts.end());
  std::string key;
  for (const auto& f : fs) key += f + ",";
  key += "->";
  for (const auto& f : fetches) key += f + ",";
  key += "/";
  for (const auto& t : ts) key += t + ",";
  auto it = executors_.find(key);
  if (it != executors_.end()) {
    *out = it->second.get();
    return Status::OK();
  }

  std::unique_ptr<ExecutorsAndKeys> ek(new ExecutorsAndKeys);
  // feeds: (node, slot) -> feed index
  std::map<std::pair<int, int>, int> feed_of;
  for (size_t i = 0; i < feeds.size(); ++i) {
    std::string node;
    int slot;
    TF_RETURN_IF_ERROR(ParseTensorName(feeds[i], &node, &slot));
    auto n = node_index_.find(node);
    if (n == node_index_.end())
      return errors::NotFound("FeedInputs: unable to find feed output ", feeds[i]);
    feed_of[{n->second, slot}] = static_cast<int>(i);
  }
  // prune: reverse reachability from fetches + targets, not expanding through fed tensors
  std::vector<int> state(nodes_.size(), 0);  // 0 unvisited, 1 in progress, 2 done
  std::vector<int> order;
  std::function<Status(int)> visit = [&](int n) -> Status {
    if (state[n] == 2) return Status::OK();
    if (state[n] == 1)
      return errors::InvalidArgument("Graph has a cycle through node '", nodes_[n]->def.name,
                                     "' (control-flow loops are outside the hot path)");
    if (!nodes_[n]->unsupported.empty()) return errors::NotFound(nodes_[n]->unsupported);
    state[n] = 1;
    for (const TensorId& in : nodes_[n]->inputs)
      if (!feed_of.count({in.node, in.slot})) TF_RETURN_IF_ERROR(visit(in.node));
    for (int c : nodes_[n]->control_inputs) TF_RETURN_IF_ERROR(visit(c));
    state[n] = 2;
    order.push_back(n);
    return Status::OK();
  };
  std::vector<TensorId> fetch_ids;
  for (const std::string& f : fetches) {
    std::string node;
    int slot;
    TF_RETURN_IF_ERROR(ParseTensorName(f, &node, &slot));
    auto n = node_index_.find(node);
    if (n == node_index_.end())
      return errors::NotFound("FetchOutputs node ", f, ": not found");
    fetch_ids.push_back(TensorId{n->second, slot});
    if (!feed_of.count({n->second, slot})) TF_RETURN_IF_ERROR(visit(n->second));
  }
  for (const std::string& t : targets) {
    auto n = node_index_.find(t);
    if (n == node_index_.end()) return errors::NotFound("Target node ", t, ": not found");
    TF_RETURN_IF_ERROR(visit(n->second));
  }
  // Schedule.  The DFS above pruned and checked for cycles; the execution order is a list
  // schedule of the pruned set: nodes in graph-construction order (the order a front-end emits
  // backprop in: last layer first); when collectives run on their own stream they are taken as
  // soon as their inputs exist, so a bucket's exchange runs under the remaining backward kernels.
  // Measured on 4 and 8 B200 (profiles/r01_notes.md): NCCL's 24-32 CTAs land on as many TPCs
  // and break up the CTA pairs of the persistent GEMMs running beside them, so the side-stream
  // exchange costs more than it hides; the default is one in-place all-reduce of the whole
  // gradient arena on the compute stream for the NCCL and peer-IPC exchanges.
  // Round 2: with the gradient arena in NVSwitch multicast memory the exchange is a 16-CTA kernel
  // whose reduction happens in the switch; it no longer disturbs the GEMMs, so on that backend the
  // overlap is the default (and captured into the step's CUDA graph).  B200TF_COLLECTIVE_OVERLAP=0 / 1
  // forces either behaviour.
  const char* ov = getenv("B200TF_COLLECTIVE_OVERLAP");
  const bool overlap_default = std::strcmp(b200_peer_arena_backend(), "nvls") == 0;
  // A plan with feeds is not graph-captured; there the side stream costs more host time than the
  // overlap returns (measured at N = 2), so it keeps the single exposed exchange.
  const bool overlap_collectives =
      device_->num_replicas() > 1 && device_->collective_comm() != nullptr &&
      (ov != nullptr ? std::strcmp(ov, "1") == 0 : (overlap_default && feeds.empty()));
  auto is_collective = [&](int n) {
    return overlap_collectives && nodes_[n]->def.op.rfind("B200AllReduce", 0) == 0 &&
           nodes_[n]->def.op != "B200AllReduce";  // the ref-variable form stays on compute
  };
  {
    std::vector<int> indeg(nodes_.size(), 0);
    std::vector<std::vector<int>> consumers(nodes_.size());
    for (int n : order) {
      for (const TensorId& in : nodes_[n]->inputs)
        if (!feed_of.count({in.node, in.slot})) {
          consumers[in.node].push_back(n);
          ++indeg[n];
        }
      for (int c : nodes_[n]->control_inputs) {
        consumers[c].push_back(n);
        ++indeg[n];
      }
    }
    typedef std::pair<int, int> Key;  // (class, node id)
    std::priority_queue<Key, std::vector<Key>, std::greater<Key>> ready;
    for (int n : order)
      if (indeg[n] == 0) ready.push(Key(is_collective(n) ? 0 : 1, n));
    std::vector<int> scheduled;
    scheduled.reserve(order.size());
    while (!ready.empty()) {
      const int n = ready.top().second;
      ready.pop();
      scheduled.push_back(n);
      for (int c : consumers[n])
        if (--indeg[c] == 0) ready.push(Key(is_collective(c) ? 0 : 1, c));
    }
    if (scheduled.size() != order.size())
      return errors::Internal("scheduler dropped nodes (", scheduled.size(), " of ", order.size(), ")");
    order.swap(scheduled);
  }
  // entry table + plan
  std::vector<int> first_entry(nodes_.size(), -1);
  for (int n : order) {
    TF_RETURN_IF_ERROR(EnsureKernel(nodes_[n].get()));
    first_entry[n] = ek->num_entries;
    ek->num_entries += std::max(1, nodes_[n]->kernel->num_outputs());
  }
  ek->entry_consumers.assign(ek->num_entries, 0);
  ek->entry_is_fetch.assign(ek->num_entries, false);
  ek->feed_needs_device.assign(feeds.size(), false);
  ek->feed_needs_host.assign(feeds.size(), false);
  for (int n : order) {
    PlanNode pn;
    pn.node = n;
    pn.item = nodes_[n].get();
    pn.first_entry = first_entry[n];
    if (is_collective(n)) {
      pn.collective = static_cast<int>(ek->collective_events.size() / 2);
      for (int e = 0; e < 2; ++e) {
        ek->collective_events.emplace_back(new gpu::Event());
        if (!ek->collective_events.back()->Init())
          return errors::Internal("could not create an event for ", nodes_[n]->def.name);
      }
    }
    const OpKernel* k = nodes_[n]->kernel.get();
    for (size_t i = 0; i < nodes_[n]->inputs.size(); ++i) {
      const TensorId& in = nodes_[n]->inputs[i];
      InputSource src;
      auto f = feed_of.find({in.node, in.slot});
      if (f != feed_of.end()) {
        src.feed = f->second;
        if (k->input_memory_types()[i] == HOST_MEMORY)
          ek->feed_needs_host[src.feed] = true;
        else
          ek->feed_needs_device[src.feed] = true;
      } else {
        src.id = in;
        const int producer_outputs = nodes_[in.node]->kernel->num_outputs();
        if (in.slot >= producer_outputs)
          return errors::InvalidArgument("Node '", nodes_[n]->def.name, "' reads output ", in.slot,
                                         " of '", nodes_[in.node]->def.name, "' which has only ",
                                         producer_outputs, " outputs");
        // dtype agreement (graph_constructor's edge type check)
        const DataType produced = nodes_[in.node]->kernel->output_type(in.slot);
        if (produced != k->input_type(i))
          return errors::InvalidArgument("Input ", i, " of node ", nodes_[n]->def.name,
                                         " was passed ", DataTypeString(produced), " from ",
                                         nodes_[in.node]->def.name, ":", in.slot,
                                         " incompatible with expected ",
                                         DataTypeString(k->input_type(i)), ".");
        ek->entry_consumers[first_entry[in.node] + in.slot]++;
      }
      pn.inputs.push_back(src);
    }
    ek->order.push_back(std::move(pn));
  }
  for (const TensorId& id : fetch_ids) {
    InputSource src;
    auto f = feed_of.find({id.node, id.slot});
    if (f != feed_of.end()) {
      src.feed = f->second;
      ek->feed_needs_host[src.feed] = true;
    } else {
      if (id.slot >= nodes_[id.node]->kernel->num_outputs())
        return errors::InvalidArgument("Fetch ", nodes_[id.node]->def.name, ":", id.slot,
                                       " is out of range");
      src.id = id;
      ek->entry_is_fetch[first_entry[id.node] + id.slot] = true;
    }
    ek->fetches.push_back(src);
  }
  ek->node_first_entry = first_entry;
  if (getenv("B200TF_DISABLE_FUSION") == nullptr) {
    TF_RETURN_IF_ERROR(FuseMatMulChains(ek.get()));
    TF_RETURN_IF_ERROR(FuseSiblingMatMuls(ek.get()));
    TF_RETURN_IF_ERROR(FuseReluGradBiasGrad(ek.get()));
    TF_RETURN_IF_ERROR(FusePoolGradReluGradBiasGrad(ek.get()));
    TF_RETURN_IF_ERROR(FuseXentScale(ek.get()));
    TF_RETURN_IF_ERROR(FuseApplyGradientDescent(ek.get()));
    // gradient buckets exist to be overlapped; exposed on the compute stream, one exchange is
    // cheaper than several (each pays the ~12 us barrier latency)
    if (!overlap_collectives) TF_RETURN_IF_ERROR(MergeAllReduceBuckets(ek.get()));
  }
  if (!EnvFlagOff("B200TF_GRADIENT_ARENA")) PlanGradientArenas(ek.get());
  *out = ek.get();
  executors_[key] = std::move(ek);
  return Status::OK();
}

void DirectSession::PlanGradientArenas(ExecutorsAndKeys* ek) {
  std::vector<std::pair<int, int>> producer_of(ek->num_entries, {-1, -1});  // entry -> (plan idx, slot)
  for (size_t p = 0; p < ek->order.size(); ++p) {
    const PlanNode& pn = ek->order[p];
    for (int o = 0; o < pn.item->kernel->num_outputs(); ++o)
      producer_of[pn.out_entry(o)] = {static_cast<int>(p), o};
  }
  for (PlanNode& pn : ek->order) {
    if (pn.item->def.op != "B200AllReduceN") continue;
    bool eligible = true;
    for (const InputSource& src : pn.inputs) {
      if (src.feed >= 0) {
        eligible = false;
        break;
      }
      const int e = entry_index_of(ek, src.id);
      const std::pair<int, int> prod = producer_of[e];
      // sole consumer, not fetched, and not already claimed by another arena
      if (ek->entry_consumers[e] != 1 || ek->entry_is_fetch[e] || prod.first < 0 ||
          (!ek->order[prod.first].arena_slots.empty() &&
           ek->order[prod.first].arena_slots[prod.second].first >= 0))
        eligible = false;
    }
    if (!eligible) continue;
    const int a = static_cast<int>(ek->arenas.size());
    ek->arenas.emplace_back();
    ek->arenas.back().dtype = pn.item->kernel->input_type(0);
    pn.arena = a;
    for (size_t i = 0; i < pn.inputs.size(); ++i) {
      const std::pair<int, int> prod = producer_of[entry_index_of(ek, pn.inputs[i].id)];
      PlanNode& producer = ek->order[prod.first];
      if (producer.arena_slots.empty())
        producer.arena_slots.assign(producer.item->kernel->num_outputs(), {-1, -1});
      producer.arena_slots[prod.second] = {a, static_cast<int>(i)};
    }
  }
}

// ReluGrad whose result feeds an NHWC BiasAddGrad (the backward pass of every conv / dense layer
// that FuseMatMulChains has not already folded into a GEMM epilogue): one node with two outputs
// that reads the gradient and the features once (`_ReluGradBiasAddGrad`).
Status DirectSession::FuseReluGradBiasGrad(ExecutorsAndKeys* ek) {
  for (size_t i = 0; i < ek->order.size(); ++i) {
    PlanNode& rg = ek->order[i];
    if (rg.dead || rg.node < 0 || rg.item->def.op != "ReluGrad") continue;
    const DataType dt = rg.item->kernel->input_type(0);
    if (dt != DT_FLOAT && dt != DT_BFLOAT16) continue;
    if (rg.inputs[0].feed >= 0 || rg.inputs[1].feed >= 0) continue;
    // the BiasAddGrad reading ReluGrad:0
    int j = -1;
    for (size_t k = i + 1; k < ek->order.size() && j < 0; ++k) {
      const PlanNode& c = ek->order[k];
      if (c.dead || c.node < 0 || c.item->def.op != "BiasAddGrad") continue;
      if (c.inputs.size() == 1 && c.inputs[0].feed < 0 && c.inputs[0].id.node == rg.node &&
          c.inputs[0].id.slot == 0)
        j = static_cast<int>(k);
    }
    if (j < 0) continue;
    PlanNode& bg = ek->order[j];
    std::string fmt = "NHWC";
    GetNodeAttr(bg.item->def, "data_format", &fmt);
    if (fmt != "NHWC") continue;
    std::unique_ptr<NodeItem> fused(new NodeItem);
    fused->def.name = bg.item->def.name + "/_relu_grad_bias_grad";
    fused->def.op = "_ReluGradBiasAddGrad";
    fused->def.attr["T"] = AttrValue::Type(dt);
    fused->def.input = {rg.item->def.input[0], rg.item->def.input[1]};
    TF_RETURN_IF_ERROR(EnsureKernel(fused.get()));
    PlanNode repl;
    repl.node = -1;
    repl.item = fused.get();
    repl.first_entry = rg.first_entry;
    repl.inputs = {rg.inputs[0], rg.inputs[1]};
    repl.output_entries = {rg.out_entry(0), bg.out_entry(0)};
    // ReluGrad:0 loses the BiasAddGrad as a consumer
    --ek->entry_consumers[rg.out_entry(0)];
    bg.dead = true;
    ek->order[i] = std::move(repl);  // at the ReluGrad's position: every consumer comes later
    ek->rewritten.push_back(std::move(fused));
  }
  std::vector<PlanNode> alive;
  for (PlanNode& pn : ek->order)
    if (!pn.dead) alive.push_back(std::move(pn));
  ek->order.swap(alive);
  return Status::OK();
}

// MaxPoolGrad whose only reader is a `_ReluGradBiasAddGrad` masking with the pool's own input (the
// backward tail of conv -> bias -> relu -> max_pool: the pool's orig_input IS the Relu output):
// `_MaxPoolGradReluGradBiasAddGrad` reads that tensor once for both the window winner and the mask
// and never materialises the pool gradient.
Status DirectSession::FusePoolGradReluGradBiasGrad(ExecutorsAndKeys* ek) {
  for (size_t i = 0; i < ek->order.size(); ++i) {
    PlanNode& pg = ek->order[i];
    if (pg.dead || pg.node < 0 || pg.item->def.op != "MaxPoolGrad" || pg.inputs.size() != 3) continue;
    const DataType dt = pg.item->kernel->input_type(0);
    if (dt != DT_FLOAT && dt != DT_BFLOAT16) continue;
    if (pg.inputs[0].feed >= 0 || pg.inputs[1].feed >= 0 || pg.inputs[2].feed >= 0) continue;
    std::string fmt = "NHWC";
    GetNodeAttr(pg.item->def, "data_format", &fmt);
    if (fmt != "NHWC") continue;
    const int dx_entry = pg.out_entry(0);
    if (ek->entry_consumers[dx_entry] != 1 || ek->entry_is_fetch[dx_entry]) continue;
    // the fused ReluGrad + BiasAddGrad reading MaxPoolGrad:0 with features == the pool's input
    int j = -1;
    for (size_t k = i + 1; k < ek->order.size() && j < 0; ++k) {
      const PlanNode& c = ek->order[k];
      if (c.dead || c.item->def.op != "_ReluGradBiasAddGrad" || c.inputs.size() != 2) continue;
      if (c.inputs[0].feed < 0 && c.inputs[0].id.node == pg.node && c.inputs[0].id.slot == 0)
        j = static_cast<int>(k);
    }
    if (j < 0) continue;
    PlanNode& rb = ek->order[j];
    if (rb.inputs[1].feed >= 0 || rb.inputs[1].id.node != pg.inputs[0].id.node ||
        rb.inputs[1].id.slot != pg.inputs[0].id.slot)
      continue;
    std::unique_ptr<NodeItem> fused(new NodeItem);
    fused->def.name = rb.item->def.name + "/_pool_grad";
    fused->def.op = "_MaxPoolGradReluGradBiasAddGrad";
    fused->def.attr = pg.item->def.attr;  // T, ksize, strides, padding, data_format
    fused->def.input = pg.item->def.input;
    TF_RETURN_IF_ERROR(EnsureKernel(fused.get()));
    PlanNode repl;
    repl.node = -1;
    repl.item = fused.get();
    repl.first_entry = rb.first_entry;
    repl.inputs = pg.inputs;
    repl.output_entries = {rb.out_entry(0), rb.out_entry(1)};
    // the pool's input loses one reader (the ReluGrad's features), the pool gradient its only one
    --ek->entry_consumers[entry_index_of(ek, pg.inputs[0].id)];
    ek->entry_consumers[dx_entry] = 0;
    pg.dead = true;
    ek->order[j] = std::move(repl);  // at the ReluGrad's position: its consumers come later
    ek->rewritten.push_back(std::move(fused));
  }
  std::vector<PlanNode> alive;
  for (PlanNode& pn : ek->order)
    if (!pn.dead) alive.push_back(std::move(pn));
  ek->order.swap(alive);
  return Status::OK();
}

// Several B200AllReduceN buckets of one dtype and scale, all on the compute stream: one node that
// reduces every gradient in a single exchange, placed where the last bucket was (all inputs exist
// there; the merge is skipped if a consumer of an earlier bucket would then run too early).
Status DirectSession::MergeAllReduceBuckets(ExecutorsAndKeys* ek) {
  std::vector<size_t> buckets;
  for (size_t i = 0; i < ek->order.size(); ++i) {
    const PlanNode& pn = ek->order[i];
    if (pn.dead || pn.node < 0 || pn.collective >= 0 || pn.item->def.op != "B200AllReduceN") continue;
    bool fed = false;
    for (const InputSource& in : pn.inputs) fed = fed || in.feed >= 0;
    if (fed) continue;
    if (!buckets.empty()) {
      const NodeDef& first = ek->order[buckets.front()].item->def;
      DataType t0 = DT_INVALID, t1 = DT_INVALID;
      float s0 = 1.f, s1 = 1.f;
      GetNodeAttr(first, "T", &t0);
      GetNodeAttr(pn.item->def, "T", &t1);
      GetNodeAttr(first, "scale", &s0);
      GetNodeAttr(pn.item->def, "scale", &s1);
      if (t0 != t1 || s0 != s1) continue;
    }
    buckets.push_back(i);
  }
  if (buckets.size() < 2) return Status::OK();
  const size_t last = buckets.back();
  // no reader of an earlier bucket may sit before the merged node
  for (size_t b = 0; b + 1 < buckets.size(); ++b) {
    const int producer = ek->order[buckets[b]].node;
    for (size_t k = buckets[b] + 1; k < last; ++k) {
      if (ek->order[k].dead) continue;
      for (const InputSource& in : ek->order[k].inputs)
        if (in.feed < 0 && in.id.node == producer) return Status::OK();
    }
  }
  std::unique_ptr<NodeItem> fused(new NodeItem);
  fused->def.name = ek->order[last].item->def.name + "/_merged";
  fused->def.op = "B200AllReduceN";
  fused->def.attr = ek->order[last].item->def.attr;
  PlanNode repl;
  repl.node = -1;
  repl.first_entry = ek->order[buckets.front()].first_entry;
  for (size_t b : buckets) {
    const PlanNode& pn = ek->order[b];
    for (size_t i = 0; i < pn.inputs.size(); ++i) {
      repl.inputs.push_back(pn.inputs[i]);
      fused->def.input.push_back(pn.item->def.input[i]);
      repl.output_entries.push_back(pn.out_entry(static_cast<int>(i)));
    }
  }
  fused->def.attr["N"] = AttrValue::I(static_cast<int64>(repl.inputs.size()));
  TF_RETURN_IF_ERROR(EnsureKernel(fused.get()));
  repl.item = fused.get();
  for (size_t b = 0; b + 1 < buckets.size(); ++b) ek->order[buckets[b]].dead = true;
  ek->order[last] = std::move(repl);
  ek->rewritten.push_back(std::move(fused));
  std::vector<PlanNode> alive;
  for (PlanNode& pn : ek->order)
    if (!pn.dead) alive.push_back(std::move(pn));
  ek->order.swap(alive);
  return Status::OK();
}

Status DirectSession::FuseApplyGradientDescent(ExecutorsAndKeys* ek) {
  size_t i = 0;
  while (i < ek->order.size()) {
    // a run: ApplyGradientDescent / Const nodes only, all updates of one dtype
    std::vector<size_t> updates;
    DataType dt = DT_INVALID;
    size_t j = i;
    for (; j < ek->order.size(); ++j) {
      const PlanNode& pn = ek->order[j];
      if (pn.node < 0) break;
      if (pn.item->def.op == "Const") continue;
      if (pn.item->def.op != "ApplyGradientDescent") break;
      const DataType t = pn.item->kernel->input_type(1);
      if ((t != DT_FLOAT && t != DT_BFLOAT16) || (dt != DT_INVALID && t != dt)) break;
      bool fed = false;
      for (const InputSource& in : pn.inputs) fed = fed || in.feed >= 0;
      if (fed) break;
      dt = t;
      updates.push_back(j);
    }
    if (updates.size() < 2) {
      i = j + 1;
      continue;
    }
    const int n = static_cast<int>(updates.size());
    std::unique_ptr<NodeItem> fused(new NodeItem);
    fused->def.name = ek->order[updates.back()].item->def.name + "/_multi_apply";
    fused->def.op = "_MultiApplyGradientDescent";
    fused->def.attr["T"] = AttrValue::Type(dt);
    fused->def.attr["N"] = AttrValue::I(n);
    PlanNode repl;
    repl.node = -1;
    repl.first_entry = ek->order[updates.front()].first_entry;
    repl.inputs.resize(3 * n);
    fused->def.input.resize(3 * n);
    for (int k = 0; k < n; ++k) {
      const PlanNode& u = ek->order[updates[k]];
      for (int a = 0; a < 3; ++a) {
        repl.inputs[a * n + k] = u.inputs[a];
        fused->def.input[a * n + k] = u.item->def.input[a];
      }
      repl.output_entries.push_back(u.out_entry(0));
    }
    TF_RETURN_IF_ERROR(EnsureKernel(fused.get()));
    repl.item = fused.get();
    for (int k = 0; k + 1 < n; ++k) ek->order[updates[k]].dead = true;
    ek->order[updates.back()] = std::move(repl);  // every delta and alpha precedes the last update
    ek->rewritten.push_back(std::move(fused));
    i = j + 1;
  }
  std::vector<PlanNode> alive;
  for (PlanNode& pn : ek->order)
    if (!pn.dead) alive.push_back(std::move(pn));
  ek->order.swap(alive);
  return Status::OK();
}

Status DirectSession::FuseXentScale(ExecutorsAndKeys* ek) {
  for (size_t i = 0; i < ek->order.size(); ++i) {
    PlanNode& xent = ek->order[i];
    if (xent.dead || xent.node < 0 || xent.item->def.op != "SoftmaxCrossEntropyWithLogits") continue;
    if (xent.item->kernel->input_type(0) != DT_FLOAT) continue;  // the fused scale is fp32-only
    const int backprop = xent.out_entry(1);
    if (ek->entry_consumers[backprop] != 1 || ek->entry_is_fetch[backprop]) continue;
    // the one consumer: Mul(backprop, c) with c a one-element Const of the same type
    int j = -1;
    for (size_t k = i + 1; k < ek->order.size() && j < 0; ++k) {
      const PlanNode& c = ek->order[k];
      if (c.dead) continue;
      for (const InputSource& in : c.inputs)
        if (in.feed < 0 && in.id.node == xent.node && in.id.slot == 1) j = static_cast<int>(k);
    }
    if (j < 0) continue;
    PlanNode& mul = ek->order[j];
    if (mul.node < 0 || mul.item->def.op != "Mul" || mul.inputs.size() != 2) continue;
    if (!(mul.inputs[0].feed < 0 && mul.inputs[0].id.node == xent.node &&
          mul.inputs[0].id.slot == 1))
      continue;
    const InputSource scale = mul.inputs[1];
    if (scale.feed >= 0 || scale.id.slot != 0) continue;
    const NodeItem* cnode = nodes_[scale.id.node].get();
    auto value = cnode->def.attr.find("value");
    if (cnode->def.op != "Const" || value == cnode->def.attr.end() ||
        value->second.tensor.dtype() != DT_FLOAT || value->second.tensor.NumElements() != 1)
      continue;
    // the Const must run before the fused node, which takes the xent's place in the order
    int cpos = -1;
    for (size_t k = 0; k < ek->order.size(); ++k)
      if (!ek->order[k].dead && ek->order[k].node == scale.id.node) cpos = static_cast<int>(k);
    if (cpos < 0) continue;

    std::unique_ptr<NodeItem> fused(new NodeItem);
    fused->def.name = mul.item->def.name + "/_scaled_xent";
    fused->def.op = "_ScaledSoftmaxCrossEntropyWithLogits";
    fused->def.attr["T"] = AttrValue::Type(DT_FLOAT);
    fused->def.input = {xent.item->def.input[0], xent.item->def.input[1], "<fused>"};
    TF_RETURN_IF_ERROR(EnsureKernel(fused.get()));
    PlanNode repl;
    repl.node = -1;
    repl.item = fused.get();
    repl.first_entry = xent.first_entry;
    repl.output_entries = {xent.out_entry(0), mul.out_entry(0)};  // loss stays, scaled backprop
    repl.inputs = {xent.inputs[0], xent.inputs[1], scale};
    ek->entry_consumers[backprop] = 0;  // nobody reads the unscaled backprop any more
    mul.dead = true;
    if (cpos > static_cast<int>(i)) {  // hoist the Const (no inputs) in front of the fused node
      PlanNode c = std::move(ek->order[cpos]);
      ek->order.erase(ek->order.begin() + cpos);
      ek->order.insert(ek->order.begin() + i, std::move(c));
      ek->order[i + 1] = std::move(repl);
      ++i;
    } else {
      ek->order[i] = std::move(repl);
    }
    ek->rewritten.push_back(std::move(fused));
  }
  std::vector<PlanNode> alive;
  for (PlanNode& pn : ek->order)
    if (!pn.dead) alive.push_back(std::move(pn));
  ek->order.swap(alive);
  return Status::OK();
}

Status DirectSession::FuseMatMulChains(ExecutorsAndKeys* ek) {
  auto entry_of = [&](const PlanNode& pn, int slot) { return pn.first_entry + slot; };
  auto single_use = [&](int entry) {
    return ek->entry_consumers[entry] == 1 && !ek->entry_is_fetch[entry];
  };
  // the unique plan node (after position `from`) reading (node, 0) as its input `want_input`
  auto consumer_of = [&](size_t from, int node, int want_input) -> int {
    for (size_t j = from + 1; j < ek->order.size(); ++j) {
      const PlanNode& c = ek->order[j];
      if (c.dead) continue;
      for (size_t i = 0; i < c.inputs.size(); ++i)
        if (c.inputs[i].feed < 0 && c.inputs[i].id.node == node && c.inputs[i].id.slot == 0)
          return static_cast<int>(i) == want_input ? static_cast<int>(j) : -1;
    }
    return -1;
  };
  for (size_t i = 0; i < ek->order.size(); ++i) {
    PlanNode& mm = ek->order[i];
    if (mm.dead || mm.node < 0) continue;
    const bool is_conv = mm.item->def.op == "Conv2D";
    if (!is_conv && mm.item->def.op != "MatMul") continue;
    if (is_conv) {  // NHWC only: the fused kernels are NHWC-native
      std::string cfmt = "NHWC";
      GetNodeAttr(mm.item->def, "data_format", &cfmt);
      if (cfmt != "NHWC") continue;
    }
    const DataType dt = mm.item->kernel->input_type(0);
    if (dt != DT_FLOAT && dt != DT_BFLOAT16) continue;
    if (!single_use(entry_of(mm, 0))) continue;
    const int j = consumer_of(i, mm.node, 0);
    if (j < 0) continue;
    PlanNode& next = ek->order[j];
    if (next.node < 0) continue;
    std::vector<std::string> fused_ops;
    int last = j;
    InputSource extra;
    if (next.item->def.op == "BiasAdd") {
      std::string fmt = "NHWC";
      GetNodeAttr(next.item->def, "data_format", &fmt);
      if (fmt != "NHWC") continue;
      fused_ops = {"BiasAdd"};
      extra = next.inputs[1];
      if (single_use(entry_of(next, 0))) {
        const int k = consumer_of(j, next.node, 0);
        if (k >= 0 && ek->order[k].node >= 0 && ek->order[k].item->def.op == "Relu") {
          fused_ops.push_back("Relu");
          last = k;
        }
      }
    } else if (!is_conv && next.item->def.op == "ReluGrad") {
      fused_ops = {"ReluGrad"};
      extra = next.inputs[1];
      // features must not be the matmul output itself
      if (extra.feed < 0 && extra.id.node == mm.node) continue;
    } else {
      continue;
    }
    std::unique_ptr<NodeItem> fused(new NodeItem);
    PlanNode& tail = ek->order[last];
    fused->def.name = tail.item->def.name + (is_conv ? "/_fused_conv2d" : "/_fused_matmul");
    fused->def.op = is_conv ? "_FusedConv2D" : "_FusedMatMul";
    fused->def.attr["T"] = AttrValue::Type(dt);
    fused->def.attr["num_args"] = AttrValue::I(1);
    if (is_conv) {
      fused->def.attr["strides"] = mm.item->def.attr.at("strides");
      fused->def.attr["padding"] = mm.item->def.attr.at("padding");
      fused->def.attr["data_format"] = AttrValue::S("NHWC");
    } else {
      fused->def.attr["transpose_a"] = mm.item->def.attr.at("transpose_a");
      fused->def.attr["transpose_b"] = mm.item->def.attr.at("transpose_b");
    }
    fused->def.attr["fused_ops"] = AttrValue::ListS(fused_ops);
    fused->def.input = {mm.item->def.input[0], mm.item->def.input[1], "<fused>"};
    TF_RETURN_IF_ERROR(EnsureKernel(fused.get()));
    PlanNode repl;
    repl.node = -1;
    repl.item = fused.get();
    repl.first_entry = tail.first_entry;  // consumers of the chain's result are unchanged
    repl.inputs = {mm.inputs[0], mm.inputs[1], extra};
    mm.dead = true;
    if (last != j) next.dead = true;
    ek->order[last] = repl;
    ek->rewritten.push_back(std::move(fused));
  }
  std::vector<PlanNode> alive;
  for (PlanNode& pn : ek->order)
    if (!pn.dead) alive.push_back(std::move(pn));
  ek->order.swap(alive);
  return Status::OK();
}

// Two live MatMul / _FusedMatMul nodes of one dtype that read the same tensor and have no fed
// input -- a dense layer's dX = dY W^T (+ ReluGrad) and dW = X^T dY -- run as one _MatMulPair:
// one persistent GEMM launch in which the second product's operand fill and main loop hide the
// first one's epilogue, and the CTA pairs one product would leave idle get work.  The pair takes
// the earlier node's place, so it is formed only when every input of the later node is produced
// before that place (which also means the later node does not depend on the earlier one) and no
// node in between updates a buffer the later node reads.  Each output keeps its entry, so the
// consumers, fetches and gradient arenas of both products are unchanged.
Status DirectSession::FuseSiblingMatMuls(ExecutorsAndKeys* ek) {
  auto candidate = [&](const PlanNode& pn) {
    if (pn.dead || (pn.item->def.op != "MatMul" && pn.item->def.op != "_FusedMatMul")) return false;
    const DataType dt = pn.item->kernel->input_type(0);
    if (dt != DT_FLOAT && dt != DT_BFLOAT16) return false;
    for (const InputSource& in : pn.inputs)
      if (in.feed >= 0) return false;
    return true;
  };
  std::vector<int> producer_pos(ek->num_entries, -1);
  for (size_t p = 0; p < ek->order.size(); ++p)
    for (int o = 0; o < ek->order[p].item->kernel->num_outputs(); ++o)
      producer_pos[ek->order[p].out_entry(o)] = static_cast<int>(p);
  auto entry_of = [&](const InputSource& in) { return entry_index_of(ek, in.id); };
  for (size_t i = 0; i < ek->order.size(); ++i) {
    if (!candidate(ek->order[i])) continue;
    const PlanNode& first = ek->order[i];
    const DataType dt = first.item->kernel->input_type(0);
    for (size_t j = i + 1; j < ek->order.size(); ++j) {
      const PlanNode& second = ek->order[j];
      if (!candidate(second) || second.item->kernel->input_type(0) != dt) continue;
      bool shared = false, ready = true;
      for (int x = 0; x < 2; ++x)
        for (int y = 0; y < 2; ++y)
          shared = shared || entry_of(first.inputs[x]) == entry_of(second.inputs[y]);
      for (const InputSource& in : second.inputs)
        ready = ready && producer_pos[entry_of(in)] < static_cast<int>(i);
      if (!shared || !ready) continue;
      // a variable update or an in-place all-reduce of one of its inputs must stay before it
      bool clobbered = false;
      for (size_t k = i + 1; k < j && !clobbered; ++k) {
        const PlanNode& mid = ek->order[k];
        if (mid.dead) continue;
        for (DataType t : mid.item->kernel->input_types())
          clobbered = clobbered || static_cast<int>(t) >= 100;  // a ref input
        if (mid.item->def.op.rfind("B200AllReduce", 0) == 0)
          for (const InputSource& a : mid.inputs)
            for (const InputSource& b : second.inputs)
              clobbered = clobbered || (a.feed < 0 && entry_of(a) == entry_of(b));
      }
      if (clobbered) continue;
      std::unique_ptr<NodeItem> fused(new NodeItem);
      fused->def.name = second.item->def.name + "/_matmul_pair";
      fused->def.op = "_MatMulPair";
      fused->def.attr["T"] = AttrValue::Type(dt);
      const PlanNode* parts[2] = {&first, &second};
      PlanNode repl;
      repl.node = -1;
      repl.first_entry = first.first_entry;
      for (int q = 0; q < 2; ++q) {
        const NodeDef& d = parts[q]->item->def;
        const std::string sfx = q == 0 ? "0" : "1";
        std::vector<std::string> ops;
        GetNodeAttr(d, "fused_ops", &ops);
        fused->def.attr["transpose_a" + sfx] = d.attr.at("transpose_a");
        fused->def.attr["transpose_b" + sfx] = d.attr.at("transpose_b");
        fused->def.attr["fused_ops" + sfx] = AttrValue::ListS(ops);
        fused->def.attr["num_args" + sfx] =
            AttrValue::I(static_cast<int64>(parts[q]->inputs.size()) - 2);
        for (size_t x = 0; x < parts[q]->inputs.size(); ++x) {
          repl.inputs.push_back(parts[q]->inputs[x]);
          fused->def.input.push_back(d.input[x]);
        }
        repl.output_entries.push_back(parts[q]->out_entry(0));
      }
      TF_RETURN_IF_ERROR(EnsureKernel(fused.get()));
      repl.item = fused.get();
      ek->order[j].dead = true;
      ek->order[i] = std::move(repl);
      ek->rewritten.push_back(std::move(fused));
      break;
    }
  }
  std::vector<PlanNode> alive;
  for (PlanNode& pn : ek->order)
    if (!pn.dead) alive.push_back(std::move(pn));
  ek->order.swap(alive);
  return Status::OK();
}

Status DirectSession::Run(const std::vector<std::pair<std::string, Tensor>>& inputs,
                          const std::vector<std::string>& output_tensor_names,
                          const std::vector<std::string>& target_node_names,
                          std::vector<Tensor>* outputs) {
  std::lock_guard<std::mutex> l(mu_);
  if (closed_) return errors::Cancelled("Session has been closed.");
  if (nodes_.empty())
    return errors::FailedPrecondition("Session was not created with a graph before Run()!");
  std::vector<std::string> feed_names;
  for (const auto& kv : inputs) feed_names.push_back(kv.first);
  ExecutorsAndKeys* ek = nullptr;
  TF_RETURN_IF_ERROR(
      GetOrCreateExecutors(feed_names, output_tensor_names, target_node_names, &ek));
  ++step_id_;
  const unsigned long long launches_before = b200_launch_count();
  stats_ = RunStats();
  const auto t0 = std::chrono::steady_clock::now();
  run_start_ = t0;
  Status s = RunPlan(ek, inputs, outputs);
  stats_.host_total_us = std::chrono::duration_cast<std::chrono::microseconds>(
                             std::chrono::steady_clock::now() - t0).count();
  if (!s.ok()) device_->Sync();  // drain whatever was enqueued before reporting
  stats_.kernels_launched = static_cast<long long>(b200_launch_count() - launches_before);
  return s;
}

static Status FromAbiStatus(int rc, const char* what) {
  if (rc == 0) return Status::OK();
  return Status(static_cast<error::Code>(rc), strings::StrCat(what, ": ", b200_last_error()));
}

// ---------------------------------------------------------------- step-level CUDA graphs
// A plan is captured when nothing in it needs the host between its first and last launch: no
// feeds (their buffers change from run to run), a single replica (the peer all-reduce kernels carry
// a per-call epoch), every kernel on the compute stream, and no input that must be moved between
// host and device memory mid-plan.  B200TF_CUDA_GRAPH=0 switches it off.
bool DirectSession::GraphEligible(ExecutorsAndKeys* ek, size_t num_feeds) {
  if (ek->graph_state != 0) return ek->graph_state > 0;
  ek->graph_state = -1;
  for (const PlanNode& pn : ek->order)
    if (pn.item->def.op == "Assign") ek->has_assign = true;
  if (ek->has_assign) return false;  // an Assign may replace a buffer other plans have captured
  const char* env = getenv("B200TF_CUDA_GRAPH");
  if (env != nullptr && std::strcmp(env, "0") == 0) return false;
  if (num_feeds != 0 || ek->order.empty()) return false;
  // Replicas: the gradient exchange must be one of our own kernels (their barrier epochs live in
  // device memory, so a replay is a fresh exchange); an NCCL call is not captured.
  const bool replicas = device_->num_replicas() > 1;
  const std::string backend = b200_peer_arena_backend();
  if (replicas && (backend == "none" || device_->peer_arena() == nullptr)) return false;
  for (const PlanNode& pn : ek->order) {
    const std::string& op = pn.item->def.op;
    if (!replicas || (op != "B200AllReduce" && op != "B200AllReduceN")) continue;
    if (op == "B200AllReduce") return false;  // the single-tensor form always goes through NCCL
    const DataType dt = pn.item->kernel->input_type(0);
    if (pn.arena < 0 || !(dt == DT_FLOAT || (dt == DT_BFLOAT16 && backend == "nvls"))) return false;
  }
  // producer memory space of every entry
  std::vector<int> entry_host(ek->num_entries, 0);
  for (const PlanNode& pn : ek->order) {
    // A node on the collective stream is captured too (the event edges fork and join the second
    // stream inside the capture) as long as it is one of the arena exchanges checked above.
    if (pn.collective >= 0 && !(replicas && pn.arena >= 0 && pn.item->def.op == "B200AllReduceN"))
      return false;
    for (int o = 0; o < pn.item->kernel->num_outputs(); ++o)
      entry_host[pn.out_entry(o)] = pn.item->kernel->output_memory_types()[o] == HOST_MEMORY;
  }
  for (const PlanNode& pn : ek->order) {
    for (size_t i = 0; i < pn.inputs.size(); ++i) {
      const InputSource& src = pn.inputs[i];
      if (src.feed >= 0) return false;
      const bool want_host = pn.item->kernel->input_memory_types()[i] == HOST_MEMORY;
      if (want_host != (entry_host[entry_index_of(ek, src.id)] != 0)) return false;
    }
  }
  ek->graph_state = 1;
  return true;
}

void DirectSession::DropGraph(ExecutorsAndKeys* ek) {
  if (ek->graph_exec != nullptr) {
    device_->Sync();
    b200_graph_destroy(ek->graph_exec);
    ek->graph_exec = nullptr;
  }
  ek->graph_fetches.clear();
  ek->graph_keepalive.clear();
  Allocator* a = device_->GetAllocator(AllocatorAttributes());
  for (void* p : ek->graph_pinned) a->DeallocateRaw(p);
  ek->graph_pinned.clear();
  if (ek->graph_state == 2) {
    ek->graph_state = 1;
    ek->warm_runs = 0;
  }
}

void DirectSession::DropAllGraphs() {
  for (auto& kv : executors_) DropGraph(kv.second.get());
}

Status DirectSession::ReplayGraph(ExecutorsAndKeys* ek, std::vector<Tensor>* outputs) {
  gpu::Stream* compute = device_->compute_stream();
  TF_RETURN_IF_ERROR(FromAbiStatus(b200_graph_launch(ek->graph_exec, compute->cuda_stream()),
                                   "cudaGraphLaunch"));
  b200_note_launches(static_cast<uint64_t>(ek->graph_launches));
  b200_note_collectives(ek->graph_peer_collectives, ek->graph_nccl_collectives);
  stats_.nodes_executed += static_cast<long long>(ek->order.size());
  outputs->clear();
  outputs->resize(ek->graph_fetches.size());
  for (size_t i = 0; i < ek->graph_fetches.size(); ++i) {
    const ExecutorsAndKeys::CapturedFetch& f = ek->graph_fetches[i];
    Tensor t = f.value;
    if (f.ref != nullptr) {
      std::lock_guard<std::mutex> rl(*f.ref_mu);
      t = *f.ref;
    }
    if (f.on_host) {
      (*outputs)[i] = t;
    } else {
      TF_RETURN_IF_ERROR(device_->CopyTensorToHost(t, &(*outputs)[i]));
      stats_.d2h_bytes += static_cast<long long>(t.TotalBytes());
    }
  }
  stats_.host_enqueue_us = std::chrono::duration_cast<std::chrono::microseconds>(
                               std::chrono::steady_clock::now() - run_start_).count();
  return device_->Sync();
}

Status DirectSession::RunPlan(ExecutorsAndKeys* ek,
                              const std::vector<std::pair<std::string, Tensor>>& inputs,
                              std::vector<Tensor>* outputs) {
  // ---- step-level CUDA graph: replay, or capture this walk
  bool capturing = false;
  if (GraphEligible(ek, inputs.size()) && b200_profile_active() == 0) {
    if (ek->graph_state == 2) return ReplayGraph(ek, outputs);
    capturing = ++ek->warm_runs >= 3;  // arenas learned, allocator and lazy inits warm
  } else if (ek->has_assign) {
    DropAllGraphs();  // this plan may give a variable a new buffer
  }
  GPUBFCAllocator* bfc = nullptr;
  unsigned long long launches_at_begin = 0;
  uint64_t peer_at_begin = 0, nccl_at_begin = 0;
  if (capturing) {
    bfc = dynamic_cast<GPUBFCAllocator*>(device_->GetAllocator(AllocatorAttributes()));
    if (bfc == nullptr ||
        b200_stream_begin_capture(device_->compute_stream()->cuda_stream()) != 0) {
      capturing = false;
      ek->graph_state = -1;
    } else {
      bfc->BeginPin();
      launches_at_begin = b200_launch_count();
      b200_collective_counts(&peer_at_begin, &nccl_at_begin);
    }
  }
  // leaves capture mode on every early return of the walk below
  struct CaptureGuard {
    DirectSession* self;
    ExecutorsAndKeys* ek;
    GPUBFCAllocator* bfc;
    bool* active;
    ~CaptureGuard() {
      if (!*active) return;
      void* exec = nullptr;
      b200_stream_end_capture(self->device_->compute_stream()->cuda_stream(), &exec);
      if (exec) b200_graph_destroy(exec);
      std::vector<void*> pinned;
      bfc->EndPin(&pinned);
      for (void* p : pinned) bfc->DeallocateRaw(p);
      ek->graph_state = -1;  // a plan whose walk failed under capture is not tried again
    }
  } capture_guard{this, ek, bfc, &capturing};

  // ---- SendInputs: stage feeds where their consumers need them
  std::vector<Tensor> feed_dev(inputs.size()), feed_host(inputs.size());
  std::vector<StagedFeed> consumed_stages;  // released after the step's sync
  std::vector<Tensor> keepalive;            // tensors touched by collective-stream nodes
  gpu::Stream* compute = device_->compute_stream();
  gpu::Stream* collective = device_->collective_stream();
  Allocator* device_allocator = device_->GetAllocator(AllocatorAttributes());
  for (size_t i = 0; i < inputs.size(); ++i) {
    const Tensor& fed = inputs[i].second;
    if (fed.buffer() != nullptr && fed.buffer()->allocator() == device_allocator) {
      // a staged (device-resident) feed: no copy, only the ordering edge
      if (ek->feed_needs_host[i])
        return errors::InvalidArgument("Feed '", inputs[i].first, "' is device-resident but a ",
                                       "consumer needs it in host memory");
      auto st = staged_.find(fed.buffer());
      if (st != staged_.end()) {
        compute->ThenWaitFor(st->second.ready.get());
        consumed_stages.push_back(std::move(st->second));
        staged_.erase(st);
      }
      feed_dev[i] = fed;
      continue;
    }
    if (ek->feed_needs_host[i]) feed_host[i] = inputs[i].second;
    if (ek->feed_needs_device[i]) {
      TF_RETURN_IF_ERROR(device_->MakeTensorFromHost(inputs[i].second, &feed_dev[i]));
      stats_.h2d_bytes += static_cast<long long>(inputs[i].second.TotalBytes());
    }
  }
  std::vector<Tensor> arena_root(ek->arenas.size());  // this step's gradient arenas
  device_->ResetPeerArena();
  std::vector<Tensor> preallocated;
  std::vector<Entry> entries(ek->num_entries);
  std::vector<int> pending(ek->entry_consumers);
  std::vector<Tensor> deref_storage;     // Tensor handles for ref->value conversions
  std::vector<TensorValue> input_values;
  std::vector<Tensor> converted;         // memory-space conversions for this node
  DeviceContext* dc = device_->device_context();

  for (const PlanNode& pn : ek->order) {
    NodeItem* item = pn.item;
    OpKernel* kernel = item->kernel.get();
    input_values.clear();
    deref_storage.clear();
    converted.clear();
    deref_storage.reserve(pn.inputs.size());
    converted.reserve(pn.inputs.size());
    for (size_t i = 0; i < pn.inputs.size(); ++i) {
      const InputSource& src = pn.inputs[i];
      const bool want_host = kernel->input_memory_types()[i] == HOST_MEMORY;
      if (src.feed >= 0) {
        if (kernel->input_is_ref(i))
          return errors::InvalidArgument("Node '", item->def.name, "': input ", i,
                                         " is a reference and cannot be fed");
        // A feed may have several consumers (and the caller may still hold the buffer): hand the
        // kernel its own handle, so that forward_input_or_allocate_output() never sees an
        // exclusively owned buffer and cannot overwrite the feed in place.
        deref_storage.push_back(want_host ? feed_host[src.feed] : feed_dev[src.feed]);
        input_values.push_back(TensorValue(&deref_storage.back()));
        continue;
      }
      Entry& en = entries[entry_index_of(ek, src.id)];
      if (!en.has_value)
        return errors::Internal("Node '", item->def.name, "': input ", i, " from '",
                                nodes_[src.id.node]->def.name, ":", src.id.slot,
                                "' was never produced");
      if (kernel->input_is_ref(i)) {
        if (en.ref == nullptr)
          return errors::InvalidArgument("Node '", item->def.name, "': input ", i,
                                         " expects a reference (variable) but got a value");
        input_values.push_back(TensorValue(en.ref_mu, en.ref));
        continue;
      }
      if (en.pending != nullptr && pn.collective < 0) {
        compute->ThenWaitFor(en.pending);  // produced on the collective stream
        en.pending = nullptr;
      }
      Tensor* t = &en.val;
      const int eidx_in = entry_index_of(ek, src.id);
      if (en.ref == nullptr && (pending[eidx_in] > 1 || ek->entry_is_fetch[eidx_in])) {
        // Other plan nodes still have to read this entry, or it is fetched: the reference gives
        // every edge its own Tensor (executor.cc Entry copies), so a kernel that forwards an
        // input in place (Relu, BiasAdd, ReluGrad ...) only ever does so for a buffer nobody else
        // will read.  Here the entry is shared, so the extra handle keeps RefCountIsOne() false.
        deref_storage.push_back(en.val);
        t = &deref_storage.back();
      }
      if (en.ref != nullptr) {  // dereference a variable for a by-value consumer
        std::lock_guard<std::mutex> rl(*en.ref_mu);
        deref_storage.push_back(*en.ref);
        t = &deref_storage.back();
        if (!t->IsInitialized() || t->NumElements() == 0)
          return errors::FailedPrecondition("Attempting to use uninitialized value ",
                                            nodes_[src.id.node]->def.name);
      }
      if (want_host != en.on_host && t->NumElements() > 0) {
        Tensor c;
        if (want_host) {  // device -> host needs the data now: sync (rare: shape-like operands)
          TF_RETURN_IF_ERROR(device_->CopyTensorToHost(*t, &c));
          TF_RETURN_IF_ERROR(device_->Sync());
          stats_.d2h_bytes += static_cast<long long>(t->TotalBytes());
        } else {
          TF_RETURN_IF_ERROR(device_->MakeTensorFromHost(*t, &c));
          stats_.h2d_bytes += static_cast<long long>(t->TotalBytes());
        }
        converted.push_back(std::move(c));
        t = &converted.back();
      }
      input_values.push_back(TensorValue(t));
    }

    OpKernelContext::Params params;
    params.step_id = step_id_;
    params.op_kernel = kernel;
    params.device = device_.get();
    params.inputs = &input_values;
    params.op_device_context = dc;
    preallocated.clear();
    if (!pn.arena_slots.empty()) {  // hand the kernel its windows of the gradient arenas
      preallocated.resize(kernel->num_outputs());
      for (int o = 0; o < kernel->num_outputs(); ++o) {
        const int a = pn.arena_slots[o].first, pos = pn.arena_slots[o].second;
        if (a < 0 || !ek->arenas[a].learned) continue;
        const GradientArena& ga = ek->arenas[a];
        const size_t esize = DataTypeSize(ga.dtype);
        if (arena_root[a].buffer() == nullptr) {
          // replicas: carve the arena from the NVLink peer arena, so that its all-reduce is one
          // kernel of peer loads (b200_peer_all_reduce); otherwise (or when it is full) the BFC arena
          const bool peer_dtype =
              ga.dtype == DT_FLOAT ||
              (ga.dtype == DT_BFLOAT16 && std::strcmp(b200_peer_arena_backend(), "nvls") == 0);
          void* peer = peer_dtype ? device_->AllocatePeerArena(ga.total) : nullptr;
          if (peer != nullptr) {
            TensorBuffer* wrap = new TensorBuffer(peer, ga.total);  // not owned
            arena_root[a] = Tensor(ga.dtype, TensorShape({static_cast<int64>(ga.total / esize)}), wrap);
            wrap->Unref();
          } else {
            arena_root[a] = Tensor(device_allocator, ga.dtype,
                                   TensorShape({static_cast<int64>(ga.total / esize)}));
          }
        }
        if (arena_root[a].buffer() == nullptr || ga.bytes[pos] == 0) continue;
        TensorBuffer* window = new TensorBuffer(arena_root[a].buffer(), ga.offsets[pos], ga.bytes[pos]);
        preallocated[o] = Tensor(ga.dtype, TensorShape({static_cast<int64>(ga.bytes[pos] / esize)}),
                                 window);
        window->Unref();
      }
      params.preallocated_outputs = &preallocated;
    }
    if (pn.arena >= 0) {  // (re)learn the layout from what the producers actually delivered
      GradientArena& ga = ek->arenas[pn.arena];
      bool same = ga.learned && ga.bytes.size() == input_values.size();
      for (size_t i = 0; same && i < input_values.size(); ++i)
        same = ga.bytes[i] == input_values[i].tensor->TotalBytes();
      if (!same) {
        ga.bytes.resize(input_values.size());
        ga.offsets.resize(input_values.size());
        size_t at = 0;
        for (size_t i = 0; i < input_values.size(); ++i) {
          ga.bytes[i] = input_values[i].tensor->TotalBytes();
          ga.offsets[i] = at;
          at += (ga.bytes[i] + 255) / 256 * 256;
        }
        ga.total = at;
        ga.learned = at > 0;
      }
    }
    gpu::Event* done = nullptr;
    if (pn.collective >= 0) {
      // everything enqueued so far (the producers of the inputs, the last users of any chunk
      // the arena hands this node) precedes the node on its own stream
      gpu::Event* inputs_ready = ek->collective_events[2 * pn.collective].get();
      done = ek->collective_events[2 * pn.collective + 1].get();
      compute->ThenRecordEvent(inputs_ready);
      collective->ThenWaitFor(inputs_ready);
      params.op_device_context = device_->collective_context();
      params.record_tensor_accesses = true;
      for (const TensorValue& v : input_values)
        if (!v.is_ref() && v.tensor != nullptr) keepalive.push_back(*v.tensor);
    }
    std::vector<AllocatorAttributes> out_attrs(kernel->num_outputs());
    for (int o = 0; o < kernel->num_outputs(); ++o)
      out_attrs[o].set_on_host(kernel->output_memory_types()[o] == HOST_MEMORY);
    params.output_attr_array = out_attrs.data();
    {
      OpKernelContext ctx(&params);
      device_->Compute(kernel, &ctx);
      ++stats_.nodes_executed;
      if (!ctx.status().ok()) {
        const Status& s = ctx.status();
        return Status(s.code(), strings::StrCat(s.error_message(), "\n\t [[Node: ",
                                                SummarizeNodeDef(item->def), "]]"));
      }
      if (done != nullptr) {
        collective->ThenRecordEvent(done);
        std::vector<Tensor> temps;
        ctx.retrieve_accessed_tensors(&temps);
        for (Tensor& t : temps) keepalive.push_back(std::move(t));
        if (!collective->ok())
          return errors::Internal("collective stream failed at node ", item->def.name);
      }
      for (int o = 0; o < kernel->num_outputs(); ++o) {
        TensorValue v = ctx.release_output(o);
        Entry& out = entries[pn.out_entry(o)];
        if (v.tensor == nullptr) {
          if (ek->entry_consumers[pn.out_entry(o)] > 0 || ek->entry_is_fetch[pn.out_entry(o)])
            return errors::Internal("Missing ", o, "-th output from ", SummarizeNodeDef(item->def));
          continue;
        }
        out.has_value = true;
        out.on_host = kernel->output_memory_types()[o] == HOST_MEMORY;
        out.pending = done;
        if (done != nullptr && !v.is_ref()) keepalive.push_back(*v.tensor);
        if (v.is_ref()) {
          out.ref = v.tensor;
          out.ref_mu = v.mutex_if_ref;
        } else {
          out.val = std::move(*v.tensor);
          delete v.tensor;
        }
      }
    }
    // release inputs whose last consumer just ran (buffers go back to the arena; reuse is
    // stream-ordered, see gpu_bfc_allocator.h)
    for (const InputSource& src : pn.inputs) {
      if (src.feed >= 0) continue;
      const int eidx = entry_index_of(ek, src.id);
      if (--pending[eidx] == 0 && !ek->entry_is_fetch[eidx]) entries[eidx].val = Tensor();
    }
  }

  // the compute stream joins every collective nobody waited for, so one sync covers the step
  for (Entry& en : entries)
    if (en.pending != nullptr) {
      compute->ThenWaitFor(en.pending);
      en.pending = nullptr;
    }

  if (capturing) {
    // the walk above was recorded, not executed: instantiate, remember what the fetches read,
    // keep every buffer the recorded kernels address, then run the step by launching the graph
    capturing = false;  // the guard must not tear the capture down any more
    void* exec = nullptr;
    const int rc = b200_stream_end_capture(compute->cuda_stream(), &exec);
    std::vector<void*> pinned;
    bfc->EndPin(&pinned);
    if (rc != 0 || exec == nullptr) {
      for (void* p : pinned) bfc->DeallocateRaw(p);
      ek->graph_state = -1;
      return errors::Internal("CUDA graph capture of the step failed: ", b200_last_error());
    }
    ek->graph_exec = exec;
    ek->graph_pinned.swap(pinned);
    ek->graph_launches = static_cast<long long>(b200_launch_count() - launches_at_begin);
    uint64_t peer_now = 0, nccl_now = 0;
    b200_collective_counts(&peer_now, &nccl_now);
    ek->graph_peer_collectives = peer_now - peer_at_begin;
    ek->graph_nccl_collectives = nccl_now - nccl_at_begin;
    ek->graph_fetches.clear();
    for (size_t i = 0; i < ek->fetches.size(); ++i) {
      const InputSource& src = ek->fetches[i];
      Entry& en = entries[entry_index_of(ek, src.id)];
      ExecutorsAndKeys::CapturedFetch f;
      f.value = en.val;
      f.ref = en.ref;
      f.ref_mu = en.ref_mu;
      f.on_host = en.on_host;
      ek->graph_fetches.push_back(f);
    }
    for (Entry& en : entries)
      if (en.val.buffer() != nullptr) ek->graph_keepalive.push_back(en.val);
    for (Tensor& t : arena_root)
      if (t.buffer() != nullptr) ek->graph_keepalive.push_back(t);
    ek->graph_state = 2;
    TF_RETURN_IF_ERROR(FromAbiStatus(b200_graph_launch(exec, compute->cuda_stream()),
                                     "cudaGraphLaunch"));
  }

  // ---- RecvOutputs: device -> pinned host, then the single sync of the step
  outputs->clear();
  outputs->resize(ek->fetches.size());
  for (size_t i = 0; i < ek->fetches.size(); ++i) {
    const InputSource& src = ek->fetches[i];
    if (src.feed >= 0) {
      (*outputs)[i] = inputs[src.feed].second;
      continue;
    }
    Entry& en = entries[entry_index_of(ek, src.id)];
    if (!en.has_value)
      return errors::Internal("Fetch ", nodes_[src.id.node]->def.name, ":", src.id.slot,
                              " was never produced");
    Tensor t = en.val;
    if (en.ref != nullptr) {
      std::lock_guard<std::mutex> rl(*en.ref_mu);
      t = *en.ref;
      if (!t.IsInitialized() || t.NumElements() == 0)
        return errors::FailedPrecondition("Attempting to use uninitialized value ",
                                          nodes_[src.id.node]->def.name);
    }
    if (en.on_host) {
      (*outputs)[i] = t;
    } else {
      TF_RETURN_IF_ERROR(device_->CopyTensorToHost(t, &(*outputs)[i]));
      stats_.d2h_bytes += static_cast<long long>(t.TotalBytes());
    }
  }
  stats_.host_enqueue_us = std::chrono::duration_cast<std::chrono::microseconds>(
                               std::chrono::steady_clock::now() - run_start_).count();
  return device_->Sync();  // sync_on_finish (keepalive / consumed_stages die after it)
}

Status DirectSession::StageFeed(const Tensor& host, Tensor* staged) {
  std::lock_guard<std::mutex> l(mu_);
  if (closed_) return errors::Cancelled("Session has been closed.");
  if (host.NumElements() == 0) return errors::InvalidArgument("cannot stage an empty tensor");
  StagedFeed st;
  st.ready.reset(new gpu::Event());
  if (!st.ready->Init()) return errors::Internal("could not create the staging event");
  st.host = host;
  Tensor dev;
  TF_RETURN_IF_ERROR(device_->StageTensorFromHost(host, &dev, st.ready.get()));
  // An entry whose copy has completed has served both purposes (ordering and keeping the pinned
  // source alive): drop it, so staged tensors that are deleted without being fed leave nothing.
  for (auto it = staged_.begin(); it != staged_.end();) {
    if (it->second.ready->PollForStatus() == gpu::Event::Status::kComplete)
      it = staged_.erase(it);
    else
      ++it;
  }
  staged_[dev.buffer()] = std::move(st);  // a stale entry for a recycled buffer is replaced
  *staged = std::move(dev);
  return Status::OK();
}

}  // namespace tensorflow
