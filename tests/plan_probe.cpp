// pybind11 wrapper of the evaluation planner (cybayes_b200/csrc/plan.cpp) for tests/test_plan.py: builds plans on the
// CPU and returns them as NumPy arrays.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>
#include <stdarg.h>
#include <stdio.h>

#include <string>

#include "plan.h"

namespace py = pybind11;

static std::string g_err;
int cb::fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}

using I32 = py::array_t<int32_t, py::array::c_style | py::array::forcecast>;

static std::vector<int32_t> vec(const I32& a) { return std::vector<int32_t>(a.data(), a.data() + a.size()); }

// cfg: PlanConfig fields by name.  snapshot: None or (buf_of_node, cherry_of_node); recs: [n_recs, 2] record children.
// Returns {"error": message} or {"ops": [n, 16], "ranges": [r, 4], "launches": [l, 4], counters...}; op columns:
// node, (kind, ref, edge) of child 0 and child 1, out_buf, pf_buf, is_root, keep, stream, spill, pushed, make_rec,
// synthetic.
static py::dict build(const py::dict& cfg_in, py::object snapshot, const I32& recs_in, const I32& offsets, const I32& nodes,
                      const I32& children, int flags, int split_env) {
  cb::PlanConfig cfg{};
  for (auto item : cfg_in) {
    const std::string k = py::str(item.first);
    py::handle v = item.second;
    if (k == "n_taxa") cfg.n_taxa = v.cast<int>();
    else if (k == "n_cats") cfg.n_cats = v.cast<int>();
    else if (k == "code_bytes") cfg.code_bytes = v.cast<int>();
    else if (k == "P") cfg.P = v.cast<int64_t>();
    else if (k == "buffer_bytes") cfg.buffer_bytes = v.cast<int64_t>();
    else if (k == "sm_count") cfg.sm_count = v.cast<int>();
    else if (k == "family_s2") cfg.family_s2 = v.cast<bool>();
    else if (k == "dmma_rc") cfg.dmma_rc = v.cast<bool>();
    else if (k == "s2_tiled") cfg.s2_tiled = v.cast<bool>();
    else if (k == "s2t_slots") cfg.s2t_slots = v.cast<int>();
    else if (k == "s2t_bulk") cfg.s2t_bulk = v.cast<bool>();
    else if (k == "s2t_prefetch") cfg.s2t_prefetch = v.cast<bool>();
    else if (k == "s2t_small_recs") cfg.s2t_small_recs = v.cast<bool>();
    else if (k == "stream_stores") cfg.stream_stores = v.cast<bool>();
    else if (k == "tile_sites") cfg.tile_sites = v.cast<int64_t>();
    else if (k == "tile_blocks") cfg.tile_blocks = v.cast<int>();
    else if (k == "blocks_per_sm") cfg.blocks_per_sm = v.cast<int>();
    else throw py::key_error("unknown PlanConfig field " + k);
  }
  cb::Snapshot sn;
  const bool have_snap = !snapshot.is_none();
  if (have_snap) {
    auto t = snapshot.cast<py::tuple>();
    sn.buf_of_node = vec(t[0].cast<I32>());
    sn.cherry_of_node = vec(t[1].cast<I32>());
  }
  std::vector<cb::CherryRec> recs(recs_in.size() / 2);
  for (size_t r = 0; r < recs.size(); ++r) {
    recs[r].tip[0] = recs_in.data()[2 * r];
    recs[r].tip[1] = recs_in.data()[2 * r + 1];
  }
  cb::EvalPlan plan;
  plan.split_env = split_env;
  g_err.clear();
  py::dict out;
  if (cb::build_plan(cfg, have_snap ? &sn : nullptr, recs, (int)offsets.size() - 1, offsets.data(), nodes.data(),
                     children.data(), flags, plan)) {
    out["error"] = g_err;
    return out;
  }
  py::array_t<int32_t> ops({(py::ssize_t)plan.ops.size(), (py::ssize_t)16});
  auto o = ops.mutable_unchecked<2>();
  for (size_t i = 0; i < plan.ops.size(); ++i) {
    const cb::PlanOp& po = plan.ops[i];
    const int32_t row[16] = {po.node, po.ch[0].kind, po.ch[0].ref, po.ch[0].edge, po.ch[1].kind, po.ch[1].ref, po.ch[1].edge,
                             po.out_buf, po.pf_buf, po.is_root, po.keep, po.stream, po.spill, po.pushed, po.make_rec, po.synthetic};
    for (int k = 0; k < 16; ++k) o(i, k) = row[k];
  }
  py::array_t<int32_t> ranges({(py::ssize_t)plan.ranges.size(), (py::ssize_t)4});
  auto r = ranges.mutable_unchecked<2>();
  for (size_t i = 0; i < plan.ranges.size(); ++i) {
    r(i, 0) = plan.ranges[i].begin; r(i, 1) = plan.ranges[i].end; r(i, 2) = plan.ranges[i].out_index; r(i, 3) = plan.ranges[i].pad_;
  }
  py::array_t<int32_t> launches({(py::ssize_t)plan.launches.size(), (py::ssize_t)4});
  auto l = launches.mutable_unchecked<2>();
  for (size_t i = 0; i < plan.launches.size(); ++i) {
    l(i, 0) = plan.launches[i].r_begin; l(i, 1) = plan.launches[i].r_end; l(i, 2) = plan.launches[i].max_ops; l(i, 3) = plan.launches[i].n_bufs;
  }
  out["ops"] = ops;
  out["ranges"] = ranges;
  out["launches"] = launches;
  out["bytes_written"] = plan.bytes_written;
  out["bytes_read"] = plan.bytes_read;
  out["n_stored"] = plan.n_stored;
  out["n_buffer_reads"] = plan.n_buffer_reads;
  out["n_stack"] = plan.n_stack;
  out["n_spills"] = plan.n_spills;
  out["n_cherries"] = plan.n_cherries;
  out["n_small_recs"] = plan.n_small_recs;
  out["n_inlined"] = plan.n_inlined;
  return out;
}

PYBIND11_MODULE(plan_probe, m) {
  m.def("build", &build);
  m.def("s2t_rank", [](int kind) { return cb::s2t_rank(kind); });
  m.def("s2t_combo", [](int k0, int k1) { return cb::s2t_combo(k0, k1); });
  m.attr("S2T_STAGING") = cb::S2T_STAGING;
  m.attr("S2T_THREADS") = cb::S2T_THREADS;
}
