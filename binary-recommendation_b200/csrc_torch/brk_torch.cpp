// PyTorch extension over the C ABI of libbrk_b200 (include/brk_b200.h): the hot-path entry points as torch custom ops
// (`torch.ops.brk.*`, TORCH_LIBRARY) taking tensors.  This is the layer BASELINE.json's north_star names -- "a PyTorch
// extension over a thin C-ABI layer standing in for the reference's framework ops" (the Keras / TFRS ops under
// /root/reference/src/models/*.py and trainers/*.py): it checks devices / dtypes / contiguity, takes the current CUDA
// stream, keeps one brk_ctx per device and forwards raw pointers.  No arithmetic lives here; there is no CPU fallback:
// a CPU tensor is an error.  The ctypes binding (_native.py) stays as the GPU-less symbol check and for the entry points
// that take structures of many tables.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <torch/types.h>

#include <mutex>
#include <unordered_map>

#include "../../include/brk_b200.h"

namespace {

std::mutex g_mu;
std::unordered_map<int, brk_ctx*> g_ctx;

// The Python side creates one brk_ctx per device through the ctypes binding; it hands the handle over so that both
// bindings share the context (workspace, tickets, copy streams).
void use_ctx(int64_t device, int64_t handle) {
  std::lock_guard<std::mutex> lock(g_mu);
  g_ctx[int(device)] = reinterpret_cast<brk_ctx*>(static_cast<intptr_t>(handle));
}

brk_ctx* ctx_for(int device) {
  std::mutex& mu = g_mu;
  std::unordered_map<int, brk_ctx*>& table = g_ctx;
  std::lock_guard<std::mutex> lock(mu);
  auto it = table.find(device);
  if (it != table.end()) return it->second;
  brk_ctx* c = nullptr;
  const int rc = brk_create(&c, device);
  TORCH_CHECK(rc == 0, "brk_create failed (rc=", rc, "): ", brk_last_error());
  table[device] = c;
  return c;
}
void check(int rc, const char* what) { TORCH_CHECK(rc == 0, what, " failed (rc=", rc, "): ", brk_last_error()); }
void need(const at::Tensor& t, at::ScalarType dt, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, ": expected a CUDA tensor (the brk hot path has no CPU fallback)");
  TORCH_CHECK(t.scalar_type() == dt, name, ": expected dtype ", dt, ", got ", t.scalar_type());
  TORCH_CHECK(t.is_contiguous(), name, ": expected a contiguous tensor");
}
void* stream_of(const at::Tensor& t) { return at::cuda::getCurrentCUDAStream(t.get_device()).stream(); }
brk_table table_of(const at::Tensor& w, const at::Tensor& g, const c10::optional<at::Tensor>& m, const c10::optional<at::Tensor>& v,
                   const c10::optional<at::Tensor>& touched) {
  need(w, at::kFloat, "w"); need(g, at::kFloat, "g");
  TORCH_CHECK(w.dim() == 2 && g.numel() == w.numel(), "table: w must be [rows, d] and g of the same size");
  brk_table t;
  t.w = w.data_ptr<float>(); t.g = g.data_ptr<float>();
  t.m = m.has_value() ? m->data_ptr<float>() : nullptr;
  t.v = v.has_value() ? v->data_ptr<float>() : nullptr;
  t.touched = touched.has_value() ? reinterpret_cast<uint32_t*>(touched->data_ptr<int32_t>()) : nullptr;
  t.rows = w.size(0); t.d = int32_t(w.size(1)); t._pad = 0;
  return t;
}

// K1: keras Embedding lookup (NeuMFModel.py:58-63, BPRModel.py:55-61, twoTower.py:34,36)
at::Tensor gather_rows(const at::Tensor& table, const at::Tensor& ids) {
  need(table, at::kFloat, "table"); need(ids, at::kInt, "ids");
  TORCH_CHECK(table.dim() == 2, "table must be [rows, d]");
  c10::cuda::CUDAGuard guard(table.device());
  at::Tensor out = at::empty({ids.numel(), table.size(1)}, table.options());
  check(brk_gather_rows(ctx_for(table.get_device()), table.data_ptr<float>(), table.size(0), int32_t(table.size(1)),
                        ids.data_ptr<int32_t>(), ids.numel(), out.data_ptr<float>(), stream_of(table)), "brk_gather_rows");
  return out;
}
// K5: IndexedSlices gradient accumulation
void scatter_add_rows(at::Tensor acc, const at::Tensor& ids, const at::Tensor& vals, const c10::optional<at::Tensor>& touched, int64_t mode) {
  need(acc, at::kFloat, "acc"); need(ids, at::kInt, "ids"); need(vals, at::kFloat, "vals");
  c10::cuda::CUDAGuard guard(acc.device());
  check(brk_scatter_add_rows(ctx_for(acc.get_device()), acc.data_ptr<float>(), acc.size(0), int32_t(acc.size(1)), ids.data_ptr<int32_t>(),
                             ids.numel(), vals.data_ptr<float>(),
                             touched.has_value() ? reinterpret_cast<uint32_t*>(touched->data_ptr<int32_t>()) : nullptr, int32_t(mode),
                             stream_of(acc)), "brk_scatter_add_rows");
}
// K10: Philox negatives of the BPR stream
at::Tensor philox_bpr_negatives(const at::Tensor& users, int64_t seed, int64_t epoch, int64_t num_items, const at::Tensor& indptr,
                                const at::Tensor& items, int64_t first_index) {
  need(users, at::kInt, "users"); need(indptr, at::kLong, "csr_indptr"); need(items, at::kInt, "csr_items");
  c10::cuda::CUDAGuard guard(users.device());
  at::Tensor out = at::empty_like(users);
  check(brk_philox_bpr_negatives(ctx_for(users.get_device()), users.data_ptr<int32_t>(), users.numel(), first_index, uint32_t(seed),
                                 uint32_t(epoch), int32_t(num_items), indptr.data_ptr<int64_t>(), items.data_ptr<int32_t>(),
                                 out.data_ptr<int32_t>(), stream_of(users)), "brk_philox_bpr_negatives");
  return out;
}
// K1+K4+K5 fused: BPR triplet forward / backward (BPRModel.py:49-74,124-144); returns the loss scalar
at::Tensor bpr_fwd_bwd(const at::Tensor& uw, at::Tensor ug, const c10::optional<at::Tensor>& ut, const at::Tensor& iw, at::Tensor ig,
                       const c10::optional<at::Tensor>& it, const at::Tensor& u, const at::Tensor& p, const at::Tensor& n, int64_t global_batch) {
  need(u, at::kInt, "u"); need(p, at::kInt, "p"); need(n, at::kInt, "n");
  c10::cuda::CUDAGuard guard(uw.device());
  const brk_table us = table_of(uw, ug, c10::nullopt, c10::nullopt, ut), is = table_of(iw, ig, c10::nullopt, c10::nullopt, it);
  at::Tensor loss = at::empty({1}, uw.options());
  check(brk_bpr_fwd_bwd(ctx_for(uw.get_device()), &us, &is, u.data_ptr<int32_t>(), p.data_ptr<int32_t>(), n.data_ptr<int32_t>(), u.numel(),
                        global_batch, loss.data_ptr<float>(), stream_of(uw)), "brk_bpr_fwd_bwd");
  return loss;
}
// K6: exact Keras Adam over a list of tables (w, g, m, v per table); state = [t, beta1^t, beta2^t] on the device
void adam_dense_keras(at::TensorList w, at::TensorList g, at::TensorList m, at::TensorList v, double lr, double b1, double b2, double eps,
                      at::Tensor state, bool advance) {
  TORCH_CHECK(w.size() == g.size() && w.size() == m.size() && w.size() == v.size() && w.size() > 0 && w.size() <= 16, "adam: 1..16 tables");
  need(state, at::kLong, "state");
  c10::cuda::CUDAGuard guard(w[0].device());
  std::vector<brk_table> tabs;
  for (size_t k = 0; k < w.size(); ++k) {
    need(m[k], at::kFloat, "m"); need(v[k], at::kFloat, "v");
    tabs.push_back(table_of(w[k].dim() == 2 ? w[k] : w[k].view({1, -1}), g[k], m[k], v[k], c10::nullopt));
  }
  brk_adam_hyper h{float(lr), float(b1), float(b2), float(eps)};
  check(brk_adam_dense_keras(ctx_for(w[0].get_device()), tabs.data(), int32_t(tabs.size()), h, state.data_ptr<int64_t>(), advance ? 1 : 0,
                             stream_of(w[0])), "brk_adam_dense_keras");
}
// K7+K8: full-catalog scoring + top-K (tfrs BruteForce: twoTower.py:64-69,229-230); bf16 rows padded to 64 columns
at::Tensor rows_to_bf16(const at::Tensor& x) {
  need(x, at::kFloat, "x");
  c10::cuda::CUDAGuard guard(x.device());
  const int32_t dpad = brk_bf16_padded_dim(int32_t(x.size(1)));
  at::Tensor out = at::empty({x.size(0), dpad}, x.options().dtype(at::kBFloat16));
  check(brk_rows_to_bf16(ctx_for(x.get_device()), x.data_ptr<float>(), x.size(0), int32_t(x.size(1)),
                         reinterpret_cast<uint16_t*>(out.data_ptr()), dpad, stream_of(x)), "brk_rows_to_bf16");
  return out;
}
std::tuple<at::Tensor, at::Tensor> score_topk(const at::Tensor& q_bf16, const at::Tensor& c_bf16, int64_t k, int64_t id_offset) {
  need(q_bf16, at::kBFloat16, "q_bf16"); need(c_bf16, at::kBFloat16, "c_bf16");
  TORCH_CHECK(q_bf16.size(1) == c_bf16.size(1), "padded widths differ");
  c10::cuda::CUDAGuard guard(q_bf16.device());
  brk_ctx* ctx = ctx_for(q_bf16.get_device());
  const int64_t U = q_bf16.size(0), I = c_bf16.size(0);
  at::Tensor vals = at::empty({U, k}, q_bf16.options().dtype(at::kFloat)), ids = at::empty({U, k}, q_bf16.options().dtype(at::kInt));
  if (U == 0) return {vals, ids};
  const int64_t wsb = brk_score_topk_workspace_bytes(ctx, U, I, int32_t(k));
  at::Tensor ws = at::empty({wsb > 16 ? wsb : 16}, q_bf16.options().dtype(at::kByte));
  check(brk_score_topk_bf16(ctx, reinterpret_cast<const uint16_t*>(q_bf16.data_ptr()), U, reinterpret_cast<const uint16_t*>(c_bf16.data_ptr()), I,
                            int32_t(q_bf16.size(1)), int32_t(k), int32_t(id_offset), vals.data_ptr<float>(), ids.data_ptr<int32_t>(),
                            ws.data_ptr(), wsb, stream_of(q_bf16)), "brk_score_topk_bf16");
  return {vals, ids};
}
// TFRS TopK.query_with_exclusions: the same selection with row r's listed global ids (CSR, ascending per row) left out
std::tuple<at::Tensor, at::Tensor> score_topk_exclude(const at::Tensor& q_bf16, const at::Tensor& c_bf16, int64_t k, int64_t id_offset,
                                                      const at::Tensor& excl_indptr, const at::Tensor& excl_ids) {
  need(q_bf16, at::kBFloat16, "q_bf16"); need(c_bf16, at::kBFloat16, "c_bf16");
  need(excl_indptr, at::kLong, "excl_indptr"); need(excl_ids, at::kInt, "excl_ids");
  TORCH_CHECK(q_bf16.size(1) == c_bf16.size(1), "padded widths differ");
  TORCH_CHECK(c_bf16.device() == q_bf16.device() && excl_indptr.device() == q_bf16.device() && excl_ids.device() == q_bf16.device(),
              "score_topk_exclude: every tensor must be on the queries' device");
  const int64_t U = q_bf16.size(0), I = c_bf16.size(0);
  TORCH_CHECK(excl_indptr.dim() == 1 && excl_indptr.numel() >= U + 1, "excl_indptr: ", excl_indptr.numel(),
              " entries, at least U + 1 = ", U + 1, " needed");
  c10::cuda::CUDAGuard guard(q_bf16.device());
  brk_ctx* ctx = ctx_for(q_bf16.get_device());
  at::Tensor vals = at::empty({U, k}, q_bf16.options().dtype(at::kFloat)), ids = at::empty({U, k}, q_bf16.options().dtype(at::kInt));
  if (U == 0) return {vals, ids};
  // an empty list array still needs an address: the C ABI takes NULL for a missing argument
  const at::Tensor xids = excl_ids.numel() ? excl_ids : at::zeros({1}, excl_ids.options());
  const int64_t wsb = brk_score_topk_workspace_bytes(ctx, U, I, int32_t(k));
  at::Tensor ws = at::empty({wsb > 16 ? wsb : 16}, q_bf16.options().dtype(at::kByte));
  check(brk_score_topk_bf16_excl(ctx, reinterpret_cast<const uint16_t*>(q_bf16.data_ptr()), U, reinterpret_cast<const uint16_t*>(c_bf16.data_ptr()),
                                 I, int32_t(q_bf16.size(1)), int32_t(k), int32_t(id_offset), excl_indptr.data_ptr<int64_t>(),
                                 xids.data_ptr<int32_t>(), vals.data_ptr<float>(), ids.data_ptr<int32_t>(), ws.data_ptr(), wsb,
                                 stream_of(q_bf16)), "brk_score_topk_bf16_excl");
  return {vals, ids};
}
std::tuple<at::Tensor, at::Tensor> topk_merge(const at::Tensor& part_vals, const at::Tensor& part_ids) {
  need(part_vals, at::kFloat, "part_vals"); need(part_ids, at::kInt, "part_ids");
  TORCH_CHECK(part_vals.dim() == 3, "part_vals must be [S, U, k]");
  c10::cuda::CUDAGuard guard(part_vals.device());
  const int64_t S = part_vals.size(0), U = part_vals.size(1), k = part_vals.size(2);
  at::Tensor vals = at::empty({U, k}, part_vals.options()), ids = at::empty({U, k}, part_ids.options());
  check(brk_topk_merge(ctx_for(part_vals.get_device()), part_vals.data_ptr<float>(), part_ids.data_ptr<int32_t>(), int32_t(S), U, int32_t(k),
                       vals.data_ptr<float>(), ids.data_ptr<int32_t>(), stream_of(part_vals)), "brk_topk_merge");
  return {vals, ids};
}
// K1..K6 fused: one NeuMF training step (model.fit's step, RModel.py:130-137).  tables: uMLP, iMLP, uMF, iMF, dense as
// parallel lists of (w, g, m, v); spec = [E, H1, H2, H3, act, loss, dropout, tensor_cores, EMF, mf_mode, no_batch_norm]
void neumf_train_step(at::TensorList w, at::TensorList g, at::TensorList m, at::TensorList v, const at::Tensor& bn_moving,
                      at::IntArrayRef spec, const at::Tensor& u, const at::Tensor& i, const at::Tensor& y, int64_t first_index,
                      int64_t dropout_seed, int64_t dropout_epoch, double lr, double b1, double b2, double eps, at::Tensor state,
                      at::Tensor ws_h1, at::Tensor ws_h2, at::Tensor ws_dy1, at::Tensor ws_dy2, at::Tensor ws_acc, at::Tensor out,
                      at::Tensor loss) {
  TORCH_CHECK(w.size() == 5 && g.size() == 5 && m.size() == 5 && v.size() == 5 && spec.size() == 11, "neumf_train_step: 5 tables, 11 spec ints");
  need(u, at::kInt, "u"); need(i, at::kInt, "i"); need(y, at::kFloat, "y"); need(state, at::kLong, "state");
  need(ws_acc, at::kDouble, "acc"); need(out, at::kFloat, "out"); need(loss, at::kFloat, "loss"); need(bn_moving, at::kFloat, "bn_moving");
  c10::cuda::CUDAGuard guard(u.device());
  brk_neumf_model mm;
  brk_table* slots[5] = {&mm.uMLP, &mm.iMLP, &mm.uMF, &mm.iMF, &mm.dense};
  for (int k = 0; k < 5; ++k) *slots[k] = table_of(w[k].dim() == 2 ? w[k] : w[k].view({1, -1}), g[k], m[k], v[k], c10::nullopt);
  mm.bn_moving = bn_moving.data_ptr<float>();
  mm.E = int32_t(spec[0]); mm.H1 = int32_t(spec[1]); mm.H2 = int32_t(spec[2]); mm.H3 = int32_t(spec[3]);
  mm.act = int32_t(spec[4]); mm.loss = int32_t(spec[5]); mm.dropout = int32_t(spec[6]); mm.tensor_cores = int32_t(spec[7]);
  mm.EMF = int32_t(spec[8]); mm.mf_mode = int32_t(spec[9]); mm.no_batch_norm = int32_t(spec[10]); mm._pad = 0;
  brk_neumf_workspace ws{ws_h1.data_ptr<float>(), ws_h2.data_ptr<float>(), ws_dy1.data_ptr<float>(), ws_dy2.data_ptr<float>(),
                         ws_acc.data_ptr<double>()};
  brk_adam_hyper h{float(lr), float(b1), float(b2), float(eps)};
  check(brk_neumf_train_step(ctx_for(u.get_device()), &mm, u.data_ptr<int32_t>(), i.data_ptr<int32_t>(), y.data_ptr<float>(), u.numel(),
                             first_index, uint32_t(dropout_seed), uint32_t(dropout_epoch), h, state.data_ptr<int64_t>(), 0, &ws,
                             out.data_ptr<float>(), loss.data_ptr<float>(), stream_of(u)), "brk_neumf_train_step");
}

int64_t abi_version() { return brk_abi_version(); }

}  // namespace

TORCH_LIBRARY(brk, m) {
  m.def("abi_version() -> int", &abi_version);
  m.def("use_ctx(int device, int handle) -> ()", &use_ctx);
  m.def("gather_rows(Tensor table, Tensor ids) -> Tensor", &gather_rows);
  m.def("scatter_add_rows(Tensor(a!) acc, Tensor ids, Tensor vals, Tensor? touched, int mode) -> ()", &scatter_add_rows);
  m.def("philox_bpr_negatives(Tensor users, int seed, int epoch, int num_items, Tensor csr_indptr, Tensor csr_items, int first_index) -> Tensor",
        &philox_bpr_negatives);
  m.def("bpr_fwd_bwd(Tensor user_w, Tensor(a!) user_g, Tensor? user_touched, Tensor item_w, Tensor(b!) item_g, Tensor? item_touched, "
        "Tensor u, Tensor p, Tensor n, int global_batch) -> Tensor", &bpr_fwd_bwd);
  m.def("adam_dense_keras(Tensor(a!)[] w, Tensor(b!)[] g, Tensor(c!)[] m, Tensor(d!)[] v, float lr, float beta1, float beta2, float eps, "
        "Tensor(e!) state, bool advance) -> ()", &adam_dense_keras);
  m.def("rows_to_bf16(Tensor x) -> Tensor", &rows_to_bf16);
  m.def("score_topk(Tensor q_bf16, Tensor c_bf16, int k, int id_offset) -> (Tensor, Tensor)", &score_topk);
  m.def("score_topk_exclude(Tensor q_bf16, Tensor c_bf16, int k, int id_offset, Tensor excl_indptr, Tensor excl_ids) -> (Tensor, Tensor)",
        &score_topk_exclude);
  m.def("topk_merge(Tensor part_vals, Tensor part_ids) -> (Tensor, Tensor)", &topk_merge);
  m.def("neumf_train_step(Tensor(a!)[] w, Tensor(b!)[] g, Tensor(c!)[] m, Tensor(d!)[] v, Tensor(e!) bn_moving, int[] spec, Tensor u, "
        "Tensor i, Tensor y, int first_index, int dropout_seed, int dropout_epoch, float lr, float beta1, float beta2, float eps, "
        "Tensor(f!) state, Tensor(g!) ws_h1, Tensor(h!) ws_h2, Tensor(i!) ws_dy1, Tensor(j!) ws_dy2, Tensor(k!) ws_acc, Tensor(l!) out, "
        "Tensor(m!) loss) -> ()", &neumf_train_step);
}
