// gc_pybind.cpp -- thin pybind11 module `medpy_b200._mgc` over the C ABI (include/medpy_b200_graphcut.h).
//
// It plays the role of the reference's Boost.Python module `medpy.graphcut.maxflow`
// (lib/maxflow/src/wrapper.cpp:59-89,125-134): one Python class owning one native graph.  Unlike the
// reference binding, whole arrays cross the boundary (numpy buffers or anything exposing
// __cuda_array_interface__, e.g. torch CUDA tensors) and the GIL is released around every native call.
// No arithmetic lives here.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <thread>
#include <string>
#include <vector>

#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "../../include/medpy_b200_graphcut.h"
#include "host_pack.hpp"

namespace py = pybind11;

namespace {

void check(int rc, const mgc_graph* g)
{
    if (rc == MGC_OK) return;
    std::string msg = mgc_last_error(g);
    if (msg.empty()) msg = "medpy_b200 graph-cut error " + std::to_string(rc);
    if (rc == MGC_E_ARG || rc == MGC_E_WEIGHT) throw py::value_error(msg);
    throw std::runtime_error(msg);
}

int dtype_code(const std::string& kind_size)
{
    if (kind_size == "f4") return MGC_F32;
    if (kind_size == "f8") return MGC_F64;
    if (kind_size == "u1" || kind_size == "b1") return MGC_U8;
    if (kind_size == "i2") return MGC_I16;
    if (kind_size == "i4") return MGC_I32;
    return -1;
}

// Holds the mgc_array plus whatever keeps the memory alive for the duration of the call.
struct ArrayRef {
    mgc_array a{};
    py::object keep;
    std::vector<int64_t> shape;
};

ArrayRef make_ref(const py::object& obj, int want_dtype /* -1 any */, const char* what)
{
    ArrayRef r;
    if (py::hasattr(obj, "__cuda_array_interface__")) {
        py::dict d = obj.attr("__cuda_array_interface__");
        py::tuple data = d["data"];
        r.a.data = reinterpret_cast<const void*>(data[0].cast<uintptr_t>());
        r.a.mem = MGC_MEM_DEVICE;
        std::string ts = d["typestr"].cast<std::string>();  // e.g. "<f4", "|u1", "|b1"
        r.a.dtype = dtype_code(ts.substr(1));
        py::tuple shp = d["shape"];
        for (auto s : shp) r.shape.push_back(s.cast<int64_t>());
        size_t es = (size_t)std::stoi(ts.substr(2));
        if (d.contains("strides") && !d["strides"].is_none()) {
            py::tuple st = d["strides"];
            for (size_t i = 0; i < st.size() && i < MGC_MAX_NDIM; ++i) r.a.strides[i] = st[i].cast<int64_t>();
        } else {
            int64_t acc = (int64_t)es;
            for (int i = (int)r.shape.size() - 1; i >= 0; --i) { if (i < MGC_MAX_NDIM) r.a.strides[i] = acc; acc *= r.shape[i]; }
        }
        r.keep = obj;
    } else {
        py::array arr = py::array::ensure(obj);
        if (!arr) throw py::value_error(std::string(what) + ": expected an array");
        std::string ks(1, arr.dtype().kind());
        ks += std::to_string(arr.dtype().itemsize());
        r.a.dtype = dtype_code(ks);
        r.a.data = arr.data();
        r.a.mem = MGC_MEM_HOST;
        for (py::ssize_t i = 0; i < arr.ndim(); ++i) {
            r.shape.push_back(arr.shape(i));
            if (i < MGC_MAX_NDIM) r.a.strides[i] = arr.strides(i);
        }
        r.keep = arr;
    }
    if (r.a.dtype < 0) throw py::value_error(std::string(what) + ": unsupported dtype");
    if (want_dtype >= 0 && r.a.dtype != want_dtype) throw py::value_error(std::string(what) + ": wrong dtype");
    return r;
}

class PyGraph {
public:
    PyGraph(const std::vector<int64_t>& shape, int device) : shape_(shape)
    {
        int rc = mgc_create((int32_t)shape.size(), shape.data(), device, &g_);
        if (rc != MGC_OK) { std::string m = mgc_last_error(nullptr); if (rc == MGC_E_ARG) throw py::value_error(m); throw std::runtime_error(m); }
    }
    PyGraph(const std::vector<int64_t>& shape, int64_t z0, int64_t z1, int device) : shape_(shape)
    {
        int rc = mgc_create_slab((int32_t)shape.size(), shape.data(), z0, z1, device, &g_);
        if (rc != MGC_OK) { std::string m = mgc_last_error(nullptr); if (rc == MGC_E_ARG) throw py::value_error(m); throw std::runtime_error(m); }
        shape_[0] = (z1 - z0) + (z0 > 0 ? 1 : 0) + (z1 < shape[0] ? 1 : 0);  // local extent incl. ghost planes
        owned_planes_ = z1 - z0;
    }
    ~PyGraph() { if (g_) mgc_destroy(g_); }
    PyGraph(const PyGraph&) = delete;
    PyGraph& operator=(const PyGraph&) = delete;

    void check_shape(const ArrayRef& r, const char* what) const
    {
        if (r.shape != shape_) throw py::value_error(std::string(what) + ": shape does not match the graph's lattice");
    }

    void add_regional_probability(const py::object& prob, double alpha, bool compute_f32)
    {
        ArrayRef r = make_ref(prob, -1, "probability_map");
        check_shape(r, "probability_map");
        int rc;
        { py::gil_scoped_release rel; rc = mgc_add_regional_probability(g_, &r.a, alpha, compute_f32 ? MGC_F32 : MGC_F64); }
        check(rc, g_);
    }
    void add_tweights_dense(const py::object& src, const py::object& snk)
    {
        ArrayRef a = make_ref(src, MGC_F64, "src"), b = make_ref(snk, MGC_F64, "snk");
        check_shape(a, "src"); check_shape(b, "snk");
        int rc;
        { py::gil_scoped_release rel; rc = mgc_add_tweights_dense(g_, &a.a, &b.a); }
        check(rc, g_);
    }
    void add_markers(const py::object& fg, const py::object& bg)
    {
        ArrayRef a, b;
        bool hf = !fg.is_none(), hb = !bg.is_none();
        if (hf) { a = make_ref(fg, MGC_U8, "fg_markers"); check_shape(a, "fg_markers"); }
        if (hb) { b = make_ref(bg, MGC_U8, "bg_markers"); check_shape(b, "bg_markers"); }
        int rc;
        { py::gil_scoped_release rel; rc = mgc_add_markers(g_, hf ? &a.a : nullptr, hb ? &b.a : nullptr); }
        check(rc, g_);
    }
    void add_boundary(int kind, const py::object& image, double sigma, const py::object& spacing, double norm)
    {
        ArrayRef r = make_ref(image, -1, "image");
        check_shape(r, "image");
        std::vector<double> sp;
        if (!spacing.is_none()) {
            sp = spacing.cast<std::vector<double>>();
            if (sp.size() < shape_.size()) throw py::value_error("spacing has fewer entries than the image has dimensions");
        }
        int rc;
        { py::gil_scoped_release rel; rc = mgc_add_boundary(g_, kind, &r.a, sigma, sp.empty() ? nullptr : sp.data(), norm); }
        check(rc, g_);
    }
    // everything graph_from_voxels adds, in one native call (mgc_build_voxel_graph); None = term absent, kind -1 = no boundary
    void build_voxel_graph(const py::object& prob, double alpha, bool compute_f32, int kind, const py::object& image, double sigma,
                           const py::object& spacing, double norm, const py::object& fg, const py::object& bg)
    {
        ArrayRef rp, ri, rf, rb;
        mgc_voxel_terms t{};
        t.alpha = alpha;
        t.compute_dtype = compute_f32 ? MGC_F32 : MGC_F64;
        t.boundary_kind = kind;
        t.sigma = sigma;
        t.norm = norm;
        if (!prob.is_none()) { rp = make_ref(prob, -1, "probability_map"); check_shape(rp, "probability_map"); t.prob = &rp.a; }
        if (!image.is_none()) { ri = make_ref(image, -1, "image"); check_shape(ri, "image"); t.image = &ri.a; }
        if (!fg.is_none()) { rf = make_ref(fg, MGC_U8, "fg_markers"); check_shape(rf, "fg_markers"); t.fg = &rf.a; }
        if (!bg.is_none()) { rb = make_ref(bg, MGC_U8, "bg_markers"); check_shape(rb, "bg_markers"); t.bg = &rb.a; }
        std::vector<double> sp;
        if (!spacing.is_none()) {
            sp = spacing.cast<std::vector<double>>();
            if (sp.size() < shape_.size()) throw py::value_error("spacing has fewer entries than the image has dimensions");
            t.spacing = sp.data();
        }
        // large host marker volumes cross PCIe bit-packed (packed on worker threads while the image is already uploading)
        std::unique_ptr<MarkerPacker> packer;
        void* bits[2] = {nullptr, nullptr};
        size_t n = 1;
        for (auto d : shape_) n *= (size_t)d;
        auto dense_host = [&](const ArrayRef& r) {
            if (r.a.mem != MGC_MEM_HOST) return false;
            int64_t expect = 1;
            for (int i = (int)r.shape.size() - 1; i >= 0; --i) { if (r.shape[i] > 1 && r.a.strides[i] != expect) return false; expect *= r.shape[i]; }
            return true;
        };
        const bool pack = pack_markers_ && n >= ((size_t)1 << 22) && mgc_can_fuse(g_) && kind >= 0 && (t.fg || t.bg) &&
                          (!t.fg || dense_host(rf)) && (!t.bg || dense_host(rb));
        if (pack) {
            const size_t words = (n + 31) / 32;
            for (int p = 0; p < 2; ++p)
                if ((p == 0 ? t.fg : t.bg) && mgc_host_alloc(words * 4, &bits[p]) != MGC_OK) throw std::runtime_error("pinned host allocation failed");
            packer.reset(new MarkerPacker(t.fg ? (const uint8_t*)rf.a.data : nullptr, t.bg ? (const uint8_t*)rb.a.data : nullptr,
                                          (uint32_t*)bits[0], (uint32_t*)bits[1], n));
            t.fg = nullptr; t.bg = nullptr;
            t.fg_bits = (const uint32_t*)bits[0]; t.bg_bits = (const uint32_t*)bits[1];
            t.bits_mem = MGC_MEM_HOST;
            t.bits_ready_words = reinterpret_cast<const volatile int64_t*>(&packer->ready);
        }
        int rc;
        { py::gil_scoped_release rel; rc = mgc_build_voxel_graph(g_, &t); packer.reset(); }
        for (int p = 0; p < 2; ++p) if (bits[p]) mgc_host_free(bits[p]);
        check(rc, g_);
    }
    void set_pack_markers(bool on) { pack_markers_ = on; }
    bool can_fuse() const { return mgc_can_fuse(g_) != 0; }
    void add_nweights_dense(int axis, const py::object& fwd, const py::object& bwd)
    {
        ArrayRef a = make_ref(fwd, MGC_F64, "fwd"), b = make_ref(bwd, MGC_F64, "bwd");
        check_shape(a, "fwd"); check_shape(b, "bwd");
        int rc;
        { py::gil_scoped_release rel; rc = mgc_add_nweights_dense(g_, axis, &a.a, &b.a); }
        check(rc, g_);
    }
    double maxflow()
    {
        double e = 0;
        int rc;
        { py::gil_scoped_release rel; rc = mgc_maxflow(g_, &e); }
        check(rc, g_);
        return e;
    }
    py::array_t<uint8_t> get_mask()
    {
        std::vector<py::ssize_t> shp(shape_.begin(), shape_.end());
        if (owned_planes_ >= 0) shp[0] = owned_planes_;
        size_t n = 1;
        for (auto d : shp) n *= (size_t)d;
        // pinned, pooled destination: the numpy array owns it through a capsule that returns it to the pool
        void* mem = nullptr;
        if (mgc_host_alloc(n ? n : 1, &mem) != MGC_OK) throw std::runtime_error("pinned host allocation failed");
        py::capsule owner(mem, [](void* p) { mgc_host_free(p); });
        int rc;
        { py::gil_scoped_release rel; rc = mgc_get_mask(g_, (uint8_t*)mem, MGC_MEM_HOST); }
        check(rc, g_);
        return py::array_t<uint8_t>(shp, (const uint8_t*)mem, owner);
    }
    void get_mask_into(uintptr_t device_ptr)
    {
        int rc;
        { py::gil_scoped_release rel; rc = mgc_get_mask(g_, reinterpret_cast<uint8_t*>(device_ptr), MGC_MEM_DEVICE); }
        check(rc, g_);
    }
    int what_segment(int64_t i) { int32_t s = 0; check(mgc_what_segment(g_, i, &s), g_); return s; }
    double get_edge(int64_t i, int64_t j) { double c = 0; check(mgc_get_edge(g_, i, j, &c), g_); return c; }
    double get_trcap(int64_t i) { double c = 0; check(mgc_get_trcap(g_, i, &c), g_); return c; }
    int64_t get_node_num() { int64_t n = 0; check(mgc_get_node_num(g_, &n), g_); return n; }
    int64_t get_arc_num() { int64_t n = 0; check(mgc_get_arc_num(g_, &n), g_); return n; }
    void reset() { check(mgc_reset(g_), g_); }
    void set_option(int option, long long value) { check(mgc_set_option(g_, option, value), g_); }
    void check_deferred() { int rc; { py::gil_scoped_release rel; rc = mgc_check(g_); } check(rc, g_); }
    void set_stream(uintptr_t s) { check(mgc_set_stream(g_, reinterpret_cast<void*>(s)), g_); }
    void synchronize() { int rc; { py::gil_scoped_release rel; rc = mgc_synchronize(g_); } check(rc, g_); }
    py::dict stats()
    {
        mgc_stats s{};
        check(mgc_get_stats(g_, &s), g_);
        py::dict d;
        d["n_voxels"] = s.n_voxels; d["push_sweeps"] = s.push_sweeps; d["global_relabels"] = s.global_relabels;
        d["relabel_sweeps"] = s.relabel_sweeps; d["kernel_launches"] = s.kernel_launches; d["active_last"] = s.active_last;
        d["ms_terms"] = s.ms_terms; d["ms_solve"] = s.ms_solve; d["ms_readout"] = s.ms_readout;
        d["ms_push"] = s.ms_push; d["ms_relabel"] = s.ms_relabel; d["ms_boundary"] = s.ms_boundary; d["ms_init"] = s.ms_init;
        d["flow_const"] = s.flow_const; d["energy"] = s.energy; d["device_bytes"] = s.device_bytes;
        int64_t bb = 0, bm = 0;
        check(mgc_get_lazy_stats(g_, &bb, &bm), g_);
        d["build_blocks"] = bb; d["blocks_materialised"] = bm;
        return d;
    }
    // ---- z-slab stepping (device pointers as integers, e.g. torch.Tensor.data_ptr()) ----
    int64_t slab_plane_elems() { int64_t n = 0; check(mgc_slab_plane_elems(g_, &n), g_); return n; }
    void slab_begin() { int rc; { py::gil_scoped_release rel; rc = mgc_slab_begin(g_); } check(rc, g_); }
    void slab_push(int n) { int rc; { py::gil_scoped_release rel; rc = mgc_slab_push(g_, n); } check(rc, g_); }
    void slab_pack(uintptr_t hlo, uintptr_t flo, uintptr_t hhi, uintptr_t fhi)
    {
        int rc;
        { py::gil_scoped_release rel; rc = mgc_slab_pack(g_, (int32_t*)hlo, (double*)flo, (int32_t*)hhi, (double*)fhi); }
        check(rc, g_);
    }
    void slab_unpack(uintptr_t hlo, uintptr_t flo, uintptr_t hhi, uintptr_t fhi, uintptr_t changed_dev)
    {
        int rc;
        { py::gil_scoped_release rel; rc = mgc_slab_unpack(g_, (const int32_t*)hlo, (const double*)flo, (const int32_t*)hhi, (const double*)fhi, (int32_t*)changed_dev); }
        check(rc, g_);
    }
    void slab_count_active_dev(uintptr_t count_dev)
    {
        int rc;
        { py::gil_scoped_release rel; rc = mgc_slab_count_active_dev(g_, (unsigned long long*)count_dev); }
        check(rc, g_);
    }
    void slab_relabel_begin() { int rc; { py::gil_scoped_release rel; rc = mgc_slab_relabel_begin(g_); } check(rc, g_); }
    int slab_relabel_relax(bool want_changed)
    {
        int32_t c = 0;
        int rc;
        { py::gil_scoped_release rel; rc = mgc_slab_relabel_relax(g_, want_changed ? &c : nullptr); }
        check(rc, g_);
        return c;
    }
    int64_t slab_count_active() { int64_t a = 0; int rc; { py::gil_scoped_release rel; rc = mgc_slab_count_active(g_, &a); } check(rc, g_); return a; }
    double slab_finish() { double e = 0; int rc; { py::gil_scoped_release rel; rc = mgc_slab_finish(g_, &e); } check(rc, g_); return e; }

    // ---- native distributed solve (NCCL inside the library) ----
    static py::bytes slab_comm_unique_id()
    {
        char id[128];
        int rc = mgc_slab_comm_unique_id(id);
        if (rc != MGC_OK) throw std::runtime_error(mgc_last_error(nullptr));
        return py::bytes(id, 128);
    }
    void slab_comm_init(int rank, int world, const py::bytes& id)
    {
        std::string s = id;
        if (s.size() != 128) throw py::value_error("the NCCL unique id has 128 bytes");
        int rc;
        { py::gil_scoped_release rel; rc = mgc_slab_comm_init(g_, rank, world, s.data()); }
        check(rc, g_);
    }
    double slab_solve()
    {
        double e = 0;
        int rc;
        { py::gil_scoped_release rel; rc = mgc_slab_solve(g_, &e); }
        check(rc, g_);
        return e;
    }
    py::dict slab_solve_stats()
    {
        int64_t a = 0, b = 0, c = 0, d = 0;
        check(mgc_slab_solve_stats(g_, &a, &b, &c, &d), g_);
        py::dict out;
        out["exchanges"] = a; out["relabel_rounds"] = b; out["push_passes"] = c; out["global_relabels"] = d;
        double ph[6] = {0, 0, 0, 0, 0, 0};
        check(mgc_slab_solve_phase_ms(g_, ph), g_);
        py::dict phase;
        phase["local_bfs_ms"] = ph[0]; phase["exchange_ms"] = ph[1]; phase["stop_test_ms"] = ph[2]; phase["push_ms"] = ph[3];
        phase["readout_ms"] = ph[4]; phase["host_blocked_ms"] = ph[5];
        out["phase_ms"] = phase;
        return out;
    }

    std::vector<int64_t> shape() const { return shape_; }

private:
    mgc_graph* g_ = nullptr;
    std::vector<int64_t> shape_;
    int64_t owned_planes_ = -1;
    bool pack_markers_ = std::getenv("MEDPY_GC_PACK_MARKERS") ? std::atoi(std::getenv("MEDPY_GC_PACK_MARKERS")) != 0 : true;
};

// ---- general sparse graph (mgc_sparse_*) ------------------------------------------------------------------------
void check_sparse(int rc, const mgc_sparse* g)
{
    if (rc == MGC_OK) return;
    std::string msg = mgc_sparse_last_error(g);
    if (msg.empty()) msg = "medpy_b200 sparse graph error " + std::to_string(rc);
    if (rc == MGC_E_ARG || rc == MGC_E_WEIGHT) throw py::value_error(msg);
    throw std::runtime_error(msg);
}

class PySparse {
public:
    PySparse(int64_t n, int device)
    {
        int rc = mgc_sparse_create(n, device, &g_);
        if (rc != MGC_OK) { std::string m = mgc_sparse_last_error(nullptr); if (rc == MGC_E_ARG) throw py::value_error(m); throw std::runtime_error(m); }
    }
    ~PySparse() { if (g_) mgc_sparse_destroy(g_); }
    PySparse(const PySparse&) = delete;
    PySparse& operator=(const PySparse&) = delete;

    void sum_edges(py::array_t<int32_t, py::array::c_style | py::array::forcecast> i,
                   py::array_t<int32_t, py::array::c_style | py::array::forcecast> j,
                   py::array_t<double, py::array::c_style | py::array::forcecast> cap,
                   py::array_t<double, py::array::c_style | py::array::forcecast> rev)
    {
        const py::ssize_t m = i.size();
        if (j.size() != m || cap.size() != m || rev.size() != m) throw py::value_error("edge arrays differ in length");
        int rc;
        { py::gil_scoped_release rel; rc = mgc_sparse_sum_edges(g_, (int64_t)m, i.data(), j.data(), cap.data(), rev.data()); }
        check_sparse(rc, g_);
    }
    void add_tweights(const py::object& nodes, py::array_t<double, py::array::c_style | py::array::forcecast> src,
                      py::array_t<double, py::array::c_style | py::array::forcecast> snk)
    {
        const py::ssize_t m = src.size();
        if (snk.size() != m) throw py::value_error("t-weight arrays differ in length");
        py::array_t<int32_t, py::array::c_style | py::array::forcecast> nd;
        const int32_t* np_ = nullptr;
        if (!nodes.is_none()) {
            nd = py::array_t<int32_t, py::array::c_style | py::array::forcecast>::ensure(nodes);
            if (!nd || nd.size() != m) throw py::value_error("node array does not match the t-weight arrays");
            np_ = nd.data();
        }
        int rc;
        { py::gil_scoped_release rel; rc = mgc_sparse_add_tweights(g_, (int64_t)m, np_, src.data(), snk.data()); }
        check_sparse(rc, g_);
    }
    double maxflow()
    {
        double e = 0;
        int rc;
        { py::gil_scoped_release rel; rc = mgc_sparse_maxflow(g_, &e); }
        check_sparse(rc, g_);
        return e;
    }
    py::array_t<uint8_t> get_mask()
    {
        int64_t n = 0;
        check_sparse(mgc_sparse_get_node_num(g_, &n), g_);
        py::array_t<uint8_t> out((py::ssize_t)n);
        int rc;
        { uint8_t* p = out.mutable_data(); py::gil_scoped_release rel; rc = mgc_sparse_get_mask(g_, p); }
        check_sparse(rc, g_);
        return out;
    }
    int what_segment(int64_t i) { int32_t s = 0; check_sparse(mgc_sparse_what_segment(g_, i, &s), g_); return s; }
    double get_edge(int64_t i, int64_t j) { double c = 0; check_sparse(mgc_sparse_get_edge(g_, i, j, &c), g_); return c; }
    double get_trcap(int64_t i) { double c = 0; check_sparse(mgc_sparse_get_trcap(g_, i, &c), g_); return c; }
    int64_t get_node_num() { int64_t n = 0; check_sparse(mgc_sparse_get_node_num(g_, &n), g_); return n; }
    int64_t get_arc_num() { int64_t n = 0; check_sparse(mgc_sparse_get_arc_num(g_, &n), g_); return n; }
    void reset() { check_sparse(mgc_sparse_reset(g_), g_); }
    py::dict stats()
    {
        mgc_stats s{};
        check_sparse(mgc_sparse_get_stats(g_, &s), g_);
        py::dict d;
        d["n_nodes"] = s.n_voxels; d["push_sweeps"] = s.push_sweeps; d["global_relabels"] = s.global_relabels;
        d["relabel_sweeps"] = s.relabel_sweeps; d["kernel_launches"] = s.kernel_launches; d["active_last"] = s.active_last;
        d["ms_solve"] = s.ms_solve; d["flow_const"] = s.flow_const; d["energy"] = s.energy; d["device_bytes"] = s.device_bytes;
        return d;
    }

private:
    mgc_sparse* g_ = nullptr;
};

// ---- label image resident on the device (mgc_labels_*) ------------------------------------------------------------
class PyLabels {
public:
    PyLabels(const py::object& labels, int device)
    {
        ArrayRef r = make_ref(labels, MGC_I32, "label_image");
        if (r.shape.empty() || r.shape.size() > MGC_MAX_NDIM) throw py::value_error("label_image must have 1 to 4 dimensions");
        shape_ = r.shape;
        int rc;
        { py::gil_scoped_release rel; rc = mgc_labels_create((int32_t)shape_.size(), shape_.data(), &r.a, device, &l_); }
        if (rc != MGC_OK) {
            std::string m = mgc_labels_last_error(nullptr);
            if (rc == MGC_E_LABELS) { PyErr_SetString(PyExc_AttributeError, m.c_str()); throw py::error_already_set(); }
            if (rc == MGC_E_ARG) throw py::value_error(m);
            throw std::runtime_error(m);
        }
    }
    ~PyLabels() { if (l_) mgc_labels_destroy(l_); }
    PyLabels(const PyLabels&) = delete;
    PyLabels& operator=(const PyLabels&) = delete;

    void check(int rc) const
    {
        if (rc == MGC_OK) return;
        std::string msg = mgc_labels_last_error(l_);
        if (msg.empty()) msg = "medpy_b200 label image error " + std::to_string(rc);
        if (rc == MGC_E_ARG) throw py::value_error(msg);
        throw std::runtime_error(msg);
    }
    ArrayRef ref(const py::object& a, int want, const char* what) const
    {
        ArrayRef r = make_ref(a, want, what);
        if (r.shape != shape_) throw py::value_error(std::string(what) + ": shape does not match the label image");
        return r;
    }
    int64_t region_count() const { int64_t k = 0; check(mgc_labels_region_count(l_, &k)); return k; }

    // -> (i, j, w_ij, w_ji), one entry per adjacent region pair, sorted by (i, j), i < j (0-based node ids)
    py::tuple boundary(int kind, const py::object& values, double directedness)
    {
        ArrayRef r;
        const bool need = kind != MGC_LABELS_ADJACENCY;
        if (need) r = ref(values, -1, "image");
        int64_t m = 0;
        int rc;
        { py::gil_scoped_release rel; rc = mgc_labels_boundary(l_, kind, need ? &r.a : nullptr, directedness, &m); }
        check(rc);
        py::array_t<int32_t> i((py::ssize_t)m), j((py::ssize_t)m);
        py::array_t<double> w((py::ssize_t)m), wr((py::ssize_t)m);
        check(mgc_labels_fetch_edges(l_, i.mutable_data(), j.mutable_data(), w.mutable_data(), wr.mutable_data()));
        return py::make_tuple(i, j, w, wr);
    }
    py::tuple region_sums(const py::object& values, int mode)
    {
        ArrayRef r = ref(values, -1, "values");
        const int64_t k = region_count();
        py::array_t<double> sums((py::ssize_t)k);
        py::array_t<int64_t> counts((py::ssize_t)k);
        int rc;
        {
            double* ps = sums.mutable_data();
            int64_t* pc = counts.mutable_data();
            py::gil_scoped_release rel;
            rc = mgc_labels_region_sums(l_, &r.a, mode, ps, pc);
        }
        check(rc);
        return py::make_tuple(sums, counts);
    }
    py::array_t<uint8_t> region_flags(const py::object& markers)
    {
        ArrayRef r = ref(markers, MGC_U8, "markers");
        py::array_t<uint8_t> flags((py::ssize_t)region_count());
        int rc;
        { uint8_t* p = flags.mutable_data(); py::gil_scoped_release rel; rc = mgc_labels_region_flags(l_, &r.a, p); }
        check(rc);
        return flags;
    }
    py::array_t<uint8_t> apply(py::array_t<uint8_t, py::array::c_style | py::array::forcecast> per_region)
    {
        if (per_region.size() != region_count()) throw py::value_error("one value per region expected");
        std::vector<py::ssize_t> shp(shape_.begin(), shape_.end());
        py::array_t<uint8_t> out(shp);
        int rc;
        { uint8_t* p = out.mutable_data(); const uint8_t* q = per_region.data(); py::gil_scoped_release rel; rc = mgc_labels_apply(l_, q, p, MGC_MEM_HOST); }
        check(rc);
        return out;
    }
    std::vector<int64_t> shape() const { return shape_; }

private:
    mgc_labels* l_ = nullptr;
    std::vector<int64_t> shape_;
};

}  // namespace

py::array_t<float> gradient_magnitude_prewitt(const py::object& image, int device)
{
    ArrayRef r = make_ref(image, -1, "image");
    if (r.shape.empty() || r.shape.size() > 4) throw py::value_error("image must have 1 to 4 dimensions");
    std::vector<py::ssize_t> shp(r.shape.begin(), r.shape.end());
    py::array_t<float> out(shp);
    int rc;
    {
        float* p = out.mutable_data();
        py::gil_scoped_release rel;
        rc = mgc_gradient_magnitude_prewitt((int32_t)r.shape.size(), r.shape.data(), &r.a, p, MGC_MEM_HOST, device);
    }
    check(rc, nullptr);
    return out;
}

PYBIND11_MODULE(_mgc, m)
{
    m.def("trim_pools", []() { mgc_trim_pools(); }, "Return every cached device / pinned block to the driver (live graphs keep theirs).");
    m.def("gradient_magnitude_prewitt", &gradient_magnitude_prewitt, py::arg("image"), py::arg("device") = -1);
    m.doc() = "pybind11 binding of libmedpy_b200_gc (B200 voxel graph-cut C ABI)";
    m.attr("ABI_VERSION") = mgc_abi_version();
    m.attr("SOURCE") = MGC_SOURCE;
    m.attr("SINK") = MGC_SINK;
    m.attr("OPT_DEFER_WEIGHT_CHECK") = MGC_OPT_DEFER_WEIGHT_CHECK;
    m.attr("OPT_KEEP_INPUTS") = MGC_OPT_KEEP_INPUTS;
    m.attr("LABELS_ADJACENCY") = MGC_LABELS_ADJACENCY;
    m.attr("LABELS_STAWIASKI") = MGC_LABELS_STAWIASKI;
    m.attr("LABELS_STAWIASKI_DIRECTED") = MGC_LABELS_STAWIASKI_DIRECTED;
    m.attr("SUM_BINCOUNT") = MGC_SUM_BINCOUNT;
    m.attr("SUM_PAIRWISE") = MGC_SUM_PAIRWISE;
    py::class_<PySparse>(m, "SparseGraph")
        .def(py::init<int64_t, int>(), py::arg("n_nodes"), py::arg("device") = -1)
        .def("sum_edges", &PySparse::sum_edges)
        .def("add_tweights", &PySparse::add_tweights)
        .def("maxflow", &PySparse::maxflow)
        .def("get_mask", &PySparse::get_mask)
        .def("what_segment", &PySparse::what_segment)
        .def("get_edge", &PySparse::get_edge)
        .def("get_trcap", &PySparse::get_trcap)
        .def("get_node_num", &PySparse::get_node_num)
        .def("get_arc_num", &PySparse::get_arc_num)
        .def("reset", &PySparse::reset)
        .def("stats", &PySparse::stats);
    py::class_<PyLabels>(m, "LabelImage")
        .def(py::init<const py::object&, int>(), py::arg("label_image"), py::arg("device") = -1)
        .def("region_count", &PyLabels::region_count)
        .def("boundary", &PyLabels::boundary, py::arg("kind"), py::arg("values") = py::none(), py::arg("directedness") = 0.0)
        .def("region_sums", &PyLabels::region_sums)
        .def("region_flags", &PyLabels::region_flags)
        .def("apply", &PyLabels::apply)
        .def_property_readonly("shape", &PyLabels::shape);
    py::class_<PyGraph>(m, "Graph")
        .def(py::init<const std::vector<int64_t>&, int>(), py::arg("shape"), py::arg("device") = -1)
        .def(py::init<const std::vector<int64_t>&, int64_t, int64_t, int>(), py::arg("shape"), py::arg("z0"), py::arg("z1"), py::arg("device") = -1)
        .def("add_regional_probability", &PyGraph::add_regional_probability)
        .def("add_tweights_dense", &PyGraph::add_tweights_dense)
        .def("add_markers", &PyGraph::add_markers)
        .def("add_boundary", &PyGraph::add_boundary)
        .def("add_nweights_dense", &PyGraph::add_nweights_dense)
        .def("build_voxel_graph", &PyGraph::build_voxel_graph)
        .def_static("slab_comm_unique_id", &PyGraph::slab_comm_unique_id)
        .def("slab_comm_init", &PyGraph::slab_comm_init)
        .def("slab_solve", &PyGraph::slab_solve)
        .def("slab_solve_stats", &PyGraph::slab_solve_stats)
        .def("can_fuse", &PyGraph::can_fuse)
        .def("set_pack_markers", &PyGraph::set_pack_markers)
        .def("maxflow", &PyGraph::maxflow)
        .def("get_mask", &PyGraph::get_mask)
        .def("get_mask_into", &PyGraph::get_mask_into)
        .def("what_segment", &PyGraph::what_segment)
        .def("get_edge", &PyGraph::get_edge)
        .def("get_trcap", &PyGraph::get_trcap)
        .def("get_node_num", &PyGraph::get_node_num)
        .def("get_arc_num", &PyGraph::get_arc_num)
        .def("reset", &PyGraph::reset)
        .def("set_option", &PyGraph::set_option)
        .def("check_deferred", &PyGraph::check_deferred)
        .def("set_stream", &PyGraph::set_stream)
        .def("synchronize", &PyGraph::synchronize)
        .def("stats", &PyGraph::stats)
        .def("slab_plane_elems", &PyGraph::slab_plane_elems)
        .def("slab_begin", &PyGraph::slab_begin)
        .def("slab_push", &PyGraph::slab_push)
        .def("slab_pack", &PyGraph::slab_pack)
        .def("slab_unpack", &PyGraph::slab_unpack)
        .def("slab_relabel_begin", &PyGraph::slab_relabel_begin)
        .def("slab_relabel_relax", &PyGraph::slab_relabel_relax, py::arg("want_changed") = false)
        .def("slab_count_active_dev", &PyGraph::slab_count_active_dev)
        .def("slab_count_active", &PyGraph::slab_count_active)
        .def("slab_finish", &PyGraph::slab_finish)
        .def_property_readonly("shape", &PyGraph::shape);
}
