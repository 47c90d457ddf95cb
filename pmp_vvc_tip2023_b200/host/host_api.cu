// Host-level entry points of libpmp_b200 for callers without Python or CUDA of their own (include/pmp_b200.h):
// pmp_weights_load (exported .pmpw weight files), pmp_predict_host (host planes in, host PartitionMat vectors out),
// pmp_predict_stream (frames in through a callback, every QP's vectors and text out window by window),
// pmp_predict_stream_multi (the same over several handles, windows in rotation), pmp_predict_stream_ex (the same with
// decode thresholds per row), pmp_format_texts (text_batch.cu), pmp_block_stats and pmp_debug_block_groups (the reuse
// of repeated blocks, block_reuse.cu), plus pmp_destroy, which releases this layer's staging before the core handle
// teardown in csrc/api.cu.
//
// This layer only calls the core's entry points and internal functions; it lives outside csrc/ because bench.py ties
// the committed ncu traffic summary (profiles/r*_traffic.json) to a hash of the csrc/ sources, and none of those kernels
// change here.  build.py compiles csrc/api.cu with -Dpmp_destroy=pmp_destroy_core so that the exported pmp_destroy is
// the one below.
#include "host.cuh"

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>

struct pmp_handle : public pmp::Handle {};      // as in csrc/api.cu

extern "C" void pmp_destroy_core(pmp_handle *h);

namespace pmp {
namespace {

// ---- .pmpw weight files ------------------------------------------------------------------------------------------
// The parameter table of nets.cu (param_spec, the reference's state_dict order, Model_QBD.py:59-253), restated for the
// file check; pmp_vvc_tip2023_b200/netspec.py holds the same table on the Python side, and the files written from it
// load through this one in tests/test_gpu_native.py.
struct Param { std::string name; int d[4]; int nd; };

void conv(std::vector<Param> &v, const std::string &name, int co, int ci, int kh, int kw, bool bias)
{
    v.push_back({name + ".weight", {co, ci, kh, kw}, 4});
    if (bias) v.push_back({name + ".bias", {co, 0, 0, 0}, 1});
}

void resblock(std::vector<Param> &v, const std::string &p, int ci, int co, int k)
{
    conv(v, p + ".left.0", co, ci, k, k, false);
    conv(v, p + ".left.2", co, co, k, k, false);
    if (ci != co) conv(v, p + ".shortcut.0", co, ci, 1, 1, false);
}

std::vector<Param> net_params(int net)
{
    std::vector<Param> v;
    const bool luma = (net == PMP_NET_LUMA_Q || net == PMP_NET_LUMA_MSBD);
    if (net == PMP_NET_LUMA_Q || net == PMP_NET_CHROMA_Q) {
        const int cin = luma ? 1 : 3, k1 = luma ? 9 : 5, k12 = luma ? 5 : 3;
        conv(v, "conv_q1", 32, cin, k1, k1, true);
        resblock(v, "resblock_q1", 32, 64, k12);
        resblock(v, "resblock_q2", 64, 64, k12);
        resblock(v, "resblock_q3", 64, 32, 3);
        resblock(v, "resblock_q4", 128, 32, 3);
        resblock(v, "resblock_q5", 32, 32, 3);
        resblock(v, "resblock_q6", 32, 8, 3);
        conv(v, "conv_q2", 1, 8, 3, 3, true);
    } else {
        const int cin = luma ? 2 : 4, kb = luma ? 9 : 5, ks = luma ? 5 : 3;
        conv(v, "conv_b1_1", 16, cin, kb, kb, true);
        conv(v, "conv_b1_2", 8, cin, ks, kb, true);
        conv(v, "conv_b1_3", 8, cin, kb, ks, true);
        resblock(v, "trunk_M1.0", 32, 64, 5);
        for (int i = 1; i < 6; i++) resblock(v, "trunk_M1." + std::to_string(i), 64, 64, 3);
        for (int i = 0; i < 4; i++) resblock(v, "trunk_M2." + std::to_string(i), 64, 64, 3);
        for (const char *b : {"B1", "B2", "B3"}) {
            resblock(v, std::string("trunk_") + b + ".0", 64, 32, 3);
            resblock(v, std::string("trunk_") + b + ".1", 32, 16, 3);
            resblock(v, std::string("trunk_") + b + ".2", 16, 8, 3);
        }
        for (const char *b : {"B1", "B2", "B3"}) conv(v, std::string("conv_") + b, 2, 8, 3, 3, true);
        for (const char *a : {"Att1", "Att2"}) {
            resblock(v, std::string("trunk_") + a + ".0", 3, 32, 3);
            resblock(v, std::string("trunk_") + a + ".1", 32, 64, 3);
        }
    }
    return v;
}

uint64_t fnv1a64(const unsigned char *p, size_t n, uint64_t x = 0xcbf29ce484222325ull)
{
    for (size_t i = 0; i < n; i++) x = (x ^ p[i]) * 0x100000001b3ull;
    return x;
}

int weights_load(Handle *h, const char *path, int *net_out, int *wset)
{
    std::vector<unsigned char> f;
    FILE *fp = fopen(path, "rb");
    if (!fp) { set_error("%s: cannot open", path); return PMP_ERR_ARG; }
    unsigned char buf[1 << 16];
    for (size_t n; (n = fread(buf, 1, sizeof buf, fp)) > 0;) f.insert(f.end(), buf, buf + n);
    const bool read_err = ferror(fp) != 0;
    fclose(fp);
    if (read_err) { set_error("%s: read error", path); return PMP_ERR_ARG; }
    auto i32 = [&](size_t off) { int32_t v; memcpy(&v, f.data() + off, 4); return v; };
    if (f.size() < 64 || memcmp(f.data(), "PMPW0001", 8) != 0) { set_error("%s: magic is not PMPW0001", path); return PMP_ERR_ARG; }
    const int net = i32(8), n = i32(12);
    int64_t total;
    uint64_t csum;
    memcpy(&total, f.data() + 16, 8);
    memcpy(&csum, f.data() + 24, 8);
    if (net < 0 || net > 3) { set_error("%s: net kind %d is not a pmp_net", path, net); return PMP_ERR_ARG; }
    const std::vector<Param> spec = net_params(net);
    if (n != (int)spec.size()) {
        set_error("%s: tensor count %d, net kind %d has %d", path, n, net, (int)spec.size());
        return PMP_ERR_ARG;
    }
    size_t off = 64;
    int64_t want_total = 0;
    std::vector<int64_t> numel(n);
    for (int i = 0; i < n; i++) {
        const Param &ps = spec[i];
        const int len = off + 4 <= f.size() ? i32(off) : -1;
        if (len < 0 || off + 8 + (size_t)len > f.size()) { set_error("%s: file ends in record %d", path, i); return PMP_ERR_ARG; }
        if ((size_t)len != ps.name.size() || memcmp(f.data() + off + 4, ps.name.data(), len) != 0) {
            set_error("%s: record %d is named '%.*s', net kind %d expects '%s'", path, i, std::min(len, 64),
                      (const char *)f.data() + off + 4, net, ps.name.c_str());
            return PMP_ERR_ARG;
        }
        off += 4 + len;
        const int nd = i32(off);
        if (nd != ps.nd || off + 4 + 4 * (size_t)nd > f.size()) {
            set_error("%s: %s has %d dims, expected %d", path, ps.name.c_str(), nd, ps.nd);
            return PMP_ERR_ARG;
        }
        numel[i] = 1;
        for (int k = 0; k < nd; k++) {
            const int d = i32(off + 4 + 4 * k);
            if (d != ps.d[k]) {
                set_error("%s: %s dim %d is %d, expected %d", path, ps.name.c_str(), k, d, ps.d[k]);
                return PMP_ERR_ARG;
            }
            numel[i] *= d;
        }
        want_total += numel[i];
        off += 4 + 4 * (size_t)nd;
    }
    off = (off + 63) & ~(size_t)63;
    if (total != want_total) {
        set_error("%s: total %lld floats, the records hold %lld", path, (long long)total, (long long)want_total);
        return PMP_ERR_ARG;
    }
    if (f.size() != off + 4 * (size_t)total) {
        set_error("%s: file size %zu, expected %zu", path, f.size(), off + 4 * (size_t)total);
        return PMP_ERR_ARG;
    }
    if (fnv1a64(f.data() + 64, f.size() - 64) != csum) { set_error("%s: checksum mismatch", path); return PMP_ERR_ARG; }
    std::vector<const float *> ptrs(n);
    for (int i = 0; i < n; i++) {       // the data starts 64-byte aligned in the file and in the buffer's allocation
        ptrs[i] = reinterpret_cast<const float *>(f.data() + off);
        off += 4 * (size_t)numel[i];
    }
    const int rc = weights_create(h, net, ptrs.data(), numel.data(), n, wset);
    if (rc == PMP_OK && net_out) *net_out = net;
    return rc;
}

// ---- the window pipeline of pmp_predict_host, pmp_predict_stream, pmp_predict_stream_multi and _ex ----------------
// Per handle: a compute and a copy stream, their events, per window slot (double-buffered) pinned + device buffers for
// the input planes, the cut blocks and the results (values, decode flags and, when asked for, text of every (row,
// component) pair, the text byte counts and a snapshot of the saturation counter), the grouping buffer (one grouping's
// scratch, each slot's groups of both components, block_reuse.cu) with the distinct counts in pinned memory, and, used
// by the compute stream only, the work area of the per-window schedule (one chunk's float maps, the post-processed qt
// map, each row's decoded integer maps and flags, and for windows with repeats the compact blocks and one row expanded
// to block order).  Created on first use, grown to the largest window, released by pmp_destroy.  The block counters of
// pmp_block_stats live here too.
constexpr int RESULTS_MAX = 8;      // 4 rows x 2 components
constexpr int STREAM_HANDLES_MAX = 16;     // handles of one pmp_predict_stream_multi call

struct HostStage {
    cudaStream_t compute = nullptr, copy = nullptr;
    cudaEvent_t uploaded[2] = {}, finished[2] = {}, downloaded[2] = {}, computed[2][RESULTS_MAX] = {};
    char *pin_in[2] = {}, *pin_out[2] = {}, *dev_in[2] = {}, *dev_out[2] = {};
    uint8_t *dev_blocks[2] = {};
    char *dev_work = nullptr, *dev_group = nullptr;
    int *pin_count = nullptr;               // [slot][component] distinct blocks of the slot's window
    size_t in_bytes = 0, out_bytes = 0, blocks_bytes = 0, work_bytes = 0;     // in, out, blocks: per slot
    long long group_cap = 0;                // blocks the grouping buffer holds
    long long stat_blocks = 0, stat_computed = 0;       // pmp_block_stats
};

std::mutex g_stage_mu;
std::map<const Handle *, HostStage> g_stage;     // a handle is used by one thread at a time; the map by all

HostStage &stage_of(const Handle *h)
{
    std::lock_guard<std::mutex> lock(g_stage_mu);
    return g_stage[h];
}

std::vector<cudaEvent_t *> events_of(HostStage &st)
{
    std::vector<cudaEvent_t *> v;
    for (int s = 0; s < 2; s++) {
        for (cudaEvent_t *e : {&st.uploaded[s], &st.finished[s], &st.downloaded[s]}) v.push_back(e);
        for (cudaEvent_t &e : st.computed[s]) v.push_back(&e);
    }
    return v;
}

void free_buffers(HostStage &st)
{
    for (int s = 0; s < 2; s++) {
        if (st.pin_in[s]) cudaFreeHost(st.pin_in[s]);
        if (st.pin_out[s]) cudaFreeHost(st.pin_out[s]);
        if (st.dev_in[s]) cudaFree(st.dev_in[s]);
        if (st.dev_out[s]) cudaFree(st.dev_out[s]);
        if (st.dev_blocks[s]) cudaFree(st.dev_blocks[s]);
        st.pin_in[s] = st.pin_out[s] = st.dev_in[s] = st.dev_out[s] = nullptr;
        st.dev_blocks[s] = nullptr;
    }
    if (st.dev_work) cudaFree(st.dev_work);
    if (st.dev_group) cudaFree(st.dev_group);
    st.dev_work = st.dev_group = nullptr;
    st.in_bytes = st.out_bytes = st.blocks_bytes = st.work_bytes = 0;
    st.group_cap = 0;
}

// The grouping buffer for `cap` blocks.  Growing it waits for the device: work in flight may use the old one.
int ensure_group(HostStage &st, long long cap)
{
    if (cap <= st.group_cap) return PMP_OK;
    PMP_CUDA(cudaDeviceSynchronize());
    if (st.dev_group) PMP_CUDA(cudaFree(st.dev_group));
    st.dev_group = nullptr;
    st.group_cap = 0;
    PMP_CUDA(cudaMalloc((void **)&st.dev_group, group_bytes(cap)));
    st.group_cap = cap;
    return PMP_OK;
}

int ensure_stage(HostStage &st, size_t in_bytes, size_t out_bytes, size_t blocks_bytes, size_t work_bytes)
{
    if (!st.compute) {
        PMP_CUDA(cudaStreamCreateWithFlags(&st.compute, cudaStreamNonBlocking));
        PMP_CUDA(cudaStreamCreateWithFlags(&st.copy, cudaStreamNonBlocking));
        for (cudaEvent_t *e : events_of(st)) PMP_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        PMP_CUDA(cudaHostAlloc((void **)&st.pin_count, 4 * sizeof(int), cudaHostAllocDefault));
    }
    if (in_bytes <= st.in_bytes && out_bytes <= st.out_bytes && blocks_bytes <= st.blocks_bytes &&
        work_bytes <= st.work_bytes)
        return PMP_OK;
    in_bytes = std::max(in_bytes, st.in_bytes);
    out_bytes = std::max(out_bytes, st.out_bytes);
    blocks_bytes = std::max(blocks_bytes, st.blocks_bytes);
    work_bytes = std::max(work_bytes, st.work_bytes);
    free_buffers(st);       // the previous call ended synchronised: nothing in flight uses them
    for (int s = 0; s < 2; s++) {
        PMP_CUDA(cudaHostAlloc((void **)&st.pin_in[s], in_bytes, cudaHostAllocDefault));
        PMP_CUDA(cudaHostAlloc((void **)&st.pin_out[s], out_bytes, cudaHostAllocDefault));
        PMP_CUDA(cudaMalloc((void **)&st.dev_in[s], in_bytes));
        PMP_CUDA(cudaMalloc((void **)&st.dev_out[s], out_bytes));
        PMP_CUDA(cudaMalloc((void **)&st.dev_blocks[s], blocks_bytes));
    }
    PMP_CUDA(cudaMalloc((void **)&st.dev_work, work_bytes));
    st.in_bytes = in_bytes;
    st.out_bytes = out_bytes;
    st.blocks_bytes = blocks_bytes;
    st.work_bytes = work_bytes;
    return PMP_OK;
}

void release_stage(const Handle *h)
{
    HostStage st;
    {
        std::lock_guard<std::mutex> lock(g_stage_mu);
        auto it = g_stage.find(h);
        if (it == g_stage.end()) return;
        st = it->second;
        g_stage.erase(it);
    }
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    free_buffers(st);
    if (!st.compute) return;
    cudaFreeHost(st.pin_count);
    for (cudaEvent_t *e : events_of(st)) cudaEventDestroy(*e);
    cudaStreamDestroy(st.compute);
    cudaStreamDestroy(st.copy);
}

// Page-locked host memory is copied from/to directly; pageable memory goes through the pinned staging.
bool host_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// on[c]: whether ws (luma Q, luma MSBD, chroma Q, chroma MSBD) runs component c; a non-skipped pair must name weight sets
// of the right net kinds.  `first` is the index of ws[0] in the caller's array, for the message.
int check_wsets(const Handle *h, const int *ws, int first, bool on[2])
{
    for (int c = 0; c < 2; c++) {
        on[c] = !(ws[2 * c] == -1 && ws[2 * c + 1] == -1);
        for (int k = 0; on[c] && k < 2; k++) {
            auto it = h->wsets.find(ws[2 * c + k]);
            if (it == h->wsets.end() || it->second.net != 2 * c + k) {
                set_error("wsets[%d] = %d is not a weight set of net kind %d", first + 2 * c + k, ws[2 * c + k], 2 * c + k);
                return PMP_ERR_ARG;
            }
        }
    }
    return PMP_OK;
}

int saturation_error(long long events)
{
    set_error("%lld fp16 saturation events: activations left the fp16 range and the results are clamped; rerun with "
              "PMP_TC_BF16 (pmp_set_engine)", events);
    return PMP_ERR_STATE;
}

// ---- weight fingerprints (pmp_predict_stream_multi's check that every handle holds the same weights) ----------------
// FNV-1a-64 over a weight set's exact fp32 parameters as the SIMT engine holds them: every conv's name, shape, packed
// weight image and bias, in the set's name order.  Copied to the host once per (handle, weight set): ids are never
// reused within a handle (next_wset++), and pmp_destroy drops the handle's entries.
std::mutex g_fp_mu;
std::map<std::pair<const Handle *, int>, uint64_t> g_fingerprint;

int wset_fingerprint(Handle *h, int id, uint64_t *out)
{
    {
        std::lock_guard<std::mutex> lock(g_fp_mu);
        auto it = g_fingerprint.find({h, id});
        if (it != g_fingerprint.end()) { *out = it->second; return PMP_OK; }
    }
    PMP_CUDA(cudaSetDevice(h->device));
    uint64_t x = fnv1a64(nullptr, 0);
    std::vector<float> buf;
    for (const auto &kv : h->wsets.at(id).convs) {      // the caller checked that the set exists
        const ConvW &cw = kv.second;
        const int dims[4] = {cw.cout, cw.cin, cw.kh, cw.kw};
        x = fnv1a64((const unsigned char *)kv.first.data(), kv.first.size(), x);
        x = fnv1a64((const unsigned char *)dims, sizeof dims, x);
        const float *part[2] = {cw.w_simt, cw.bias};
        const size_t n[2] = {cw.w_simt ? (size_t)cw.cin * cw.kh * cw.kw * ((cw.cout + 3) & ~3) : 0,   // nets.cu's layout
                             cw.bias ? (size_t)cw.cout : 0};
        for (int p = 0; p < 2; p++) {
            buf.resize(n[p]);
            if (n[p]) PMP_CUDA(cudaMemcpy(buf.data(), part[p], n[p] * sizeof(float), cudaMemcpyDeviceToHost));
            x = fnv1a64((const unsigned char *)buf.data(), n[p] * sizeof(float), x);
        }
    }
    std::lock_guard<std::mutex> lock(g_fp_mu);
    g_fingerprint[{h, id}] = x;
    *out = x;
    return PMP_OK;
}

void release_fingerprints(const Handle *h)
{
    std::lock_guard<std::mutex> lock(g_fp_mu);
    g_fingerprint.erase(g_fingerprint.lower_bound({h, INT_MIN}), g_fingerprint.upper_bound({h, INT_MAX}));
}

// One call's work: the (row, component) results over `frames` frames, in windows of `wf` whole frames.  A row is a QP's
// weight sets and a set of decode thresholds.  The entry point supplies the host ends of a window: fill() provides its
// input planes, write() takes its results.
struct WindowJob {
    int n_qps = 0, frames = 0, width = 0, height = 0, sample_bytes = 1, wf = 1, chunk = 4800;     // n_qps: the rows
    bool on[4][2] = {};
    const double *lamb = nullptr;           // [n_qps][5] lamb1..lamb5 per row; nullptr: the reference defaults
    bool values = true, text = false;       // download the values; format and download the text
    bool stop_on_saturation = false;        // stop after the first window with saturation events, or finish them all
    bool direct_in = false;                 // fill() points src at the caller's page-locked planes and leaves pin alone
    // Frames [f0, f0 + nf): fills pin[p] (dense planes y, u, v; u and v only when a QP runs chroma) or points src[p]
    // (preset to pin[p]) at page-locked planes of the same layout.  Returns a pmp_status.
    std::function<int(int f0, int nf, char *const pin[3], const char *src[3])> fill;
    // Optional: page-locked destination of result (q, c)'s values of the window starting at f0, nullptr = the staging.
    std::function<int8_t *(int f0, int q, int c)> direct_out;
    std::function<int(const pmp_window &w)> write;      // returns a pmp_status
};

// One handle's part of a call: windows k with k % lanes == its index, on its own streams and staging.
struct Lane {
    pmp_handle *h = nullptr;
    const int *wsets = nullptr;     // [rows][4]: this handle's weight-set ids
    HostStage *st = nullptr;        // set by run_windows
    unsigned int sat_prev = 0;      // the handle's saturation counter after its previous window
};

// Runs `job` over the lanes in rotation: window k runs on lanes[k % n].  Iteration k computes window k, fills and
// uploads window k + n, downloads window k and writes window k - n, so each lane keeps both its window slots busy while
// the host reads and writes in frame order; with one lane, window k+1 is filled and uploaded and window k-1 written
// while window k computes.  Each lane's first window is computed as soon as it is uploaded, so that no device waits for
// the other lanes' first reads.  Each window is cut into blocks once for all its results, on the copy stream right after
// its upload, and each component's blocks are grouped there (block_reuse.cu): the distinct count reaches pinned memory
// behind the `uploaded` event, long before the compute stream gets to the window.  Per component, rows whose (Q, MSBD)
// weight-set ids are equal share one net pass: per chunk of job.chunk blocks, pmp_predict_maps and pmp_qt_postprocess
// run once and pmp_map2partition_ex once per row with the row's thresholds; then pmp_assemble_frames runs once per row.
// With one row per pass this is exactly the sequence of pmp_run_component.  When a component's window holds repeated
// blocks, the pass runs on its distinct blocks only: they are gathered into compact order first, and each row's decoded
// maps, flags and the qt map are expanded back to block order before pmp_assemble_frames.  Without repeats the sequence
// is the one above on the cut blocks.  The host waits only on events of finished windows and of uploads that finished
// while an earlier window computed.  The device of a lane is made current before each of its CUDA calls; fill() and write()
// may switch devices.  *total receives the sum of the reports of the windows written.  Every return leaves no work
// queued on any lane.
int run_windows(std::vector<Lane> &lanes, const WindowJob &job, pmp_report *total)
{
    memset(total, 0, sizeof(*total));
    const int bh = job.height / 64, bw = job.width / 64, bpf = bh * bw, wf = job.wf, frames = job.frames;
    const long long nmax = (long long)wf * bpf;
    const int64_t per = pmp_frame_values(bh, bw);
    int nres = 0, res_q[RESULTS_MAX], res_c[RESULTS_MAX];
    bool comp_on[2] = {false, false};
    for (int q = 0; q < job.n_qps; q++)
        for (int c = 0; c < 2; c++)
            if (job.on[q][c]) {
                res_q[nres] = q;
                res_c[nres++] = c;
                comp_on[c] = true;
            }
    const bool chroma = comp_on[1];
    const size_t row_y = (size_t)job.width * job.sample_bytes, row_c = row_y / 2;
    const size_t plane_y = (size_t)job.height * row_y, plane_c = (size_t)(job.height / 2) * row_c;
    const size_t in_frame = plane_y + (chroma ? 2 * plane_c : 0);
    const size_t rows[3] = {(size_t)job.height, (size_t)job.height / 2, (size_t)job.height / 2};
    const size_t prow[3] = {row_y, row_c, row_c};
    const int nplanes = chroma ? 3 : 1;
    auto in_off = [&](int p, int nf) { return p == 0 ? 0 : (size_t)nf * (plane_y + (p - 1) * plane_c); };
    // per slot: values, flags and text of each result, then the text byte counts and the saturation snapshot
    auto r256 = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t vals_bytes = r256((size_t)wf * per), flags_bytes = r256((size_t)nmax * 4),
                 text_bytes = job.text ? r256((size_t)3 * wf * per) : 0;
    size_t off_vals[RESULTS_MAX], off_flags[RESULTS_MAX], off_text[RESULTS_MAX], off = 0;
    for (int i = 0; i < nres; i++) {
        off_vals[i] = off;
        off_flags[i] = off += vals_bytes;
        off_text[i] = off += flags_bytes;
        off += text_bytes;
    }
    const size_t off_nbytes = off, off_sat = off + 8 * RESULTS_MAX;
    const size_t blk_bytes[2] = {(size_t)68 * 68, (size_t)3 * 34 * 34};
    // the work area: one chunk's float maps (qt [64] | bt [768] | dire [768] f32 per block), the window's
    // post-processed qt map [64] u8 per block, per row of a shared net pass hor [256] | ver [256] | dire [768] and the
    // flags [u32]; for windows with repeated blocks the compact blocks, the qt map and one row's maps in block order
    const int chunk = (int)std::min<long long>(job.chunk, nmax);
    const size_t maps_bytes = r256((size_t)chunk * (64 + 768 + 768) * sizeof(float)), qt8_bytes = r256((size_t)nmax * 64),
                 dec_bytes = r256((size_t)nmax * (256 + 256 + 768)), row_bytes = dec_bytes + r256((size_t)nmax * 4),
                 compact_bytes = r256((size_t)nmax * (comp_on[0] ? blk_bytes[0] : blk_bytes[1]));
    const size_t off_rows = maps_bytes + qt8_bytes, off_compact = off_rows + (size_t)job.n_qps * row_bytes,
                 off_qtx = off_compact + compact_bytes, off_expanded = off_qtx + qt8_bytes;
    const int nwin = (frames + wf - 1) / wf;
    if ((int)lanes.size() > nwin) lanes.resize(nwin);       // lanes without a window stay untouched
    const int n = (int)lanes.size();
    int rc = PMP_OK;
    for (Lane &ln : lanes) {
        pmp_handle *h = ln.h;
        PMP_CUDA(cudaSetDevice(h->device));
        ln.st = &stage_of(h);
        rc = ensure_stage(*ln.st, (size_t)wf * in_frame, off_sat + 256,
                          (size_t)nmax * ((comp_on[0] ? blk_bytes[0] : 0) + (comp_on[1] ? blk_bytes[1] : 0)),
                          off_expanded + dec_bytes);
        if (rc || (rc = ensure_group(*ln.st, nmax))) return rc;
        // The status word and the text status words exist before the loop (allocating them synchronises the device).
        // The activation arena grows inside the first window's pmp_predict_maps when a handle first sees this chunk
        // size; that synchronises the device once and leaves everything queued intact.
        if ((rc = ensure_status(h))) return rc;
        if (job.text && (rc = reserve_text_status(h, nres, (long long)wf * per))) return rc;
        PMP_CUDA(cudaDeviceSynchronize());
        PMP_CUDA(cudaMemcpy(&ln.sat_prev, h->d_status, sizeof(ln.sat_prev), cudaMemcpyDeviceToHost));
    }

    auto win_frames = [&](int k) { return std::min(wf, frames - k * wf); };
    auto direct = [&](int f0, int i) -> int8_t * { return job.direct_out ? job.direct_out(f0, res_q[i], res_c[i]) : nullptr; };
    auto blocks_of = [&](const HostStage &st, int s, int c) -> uint8_t * {
        return !comp_on[c] ? nullptr : st.dev_blocks[s] + (c == 1 && comp_on[0] ? (size_t)nmax * blk_bytes[0] : 0);
    };

    auto upload = [&](int k) -> int {
        Lane &ln = lanes[k % n];
        HostStage &st = *ln.st;
        const int j = k / n, s = j & 1, f0 = k * wf, nf = win_frames(k);      // j: the lane's own window count
        PMP_CUDA(cudaSetDevice(ln.h->device));
        if (j >= 2) {
            if (!job.direct_in) PMP_CUDA(cudaEventSynchronize(st.uploaded[s]));     // pin_in[s] free again
            PMP_CUDA(cudaStreamWaitEvent(st.copy, st.finished[s], 0));      // blocks and groups of slot s read by j-2
        }
        char *pin[3] = {nullptr, nullptr, nullptr};
        const char *src[3] = {nullptr, nullptr, nullptr};
        for (int p = 0; p < nplanes; p++) src[p] = pin[p] = st.pin_in[s] + in_off(p, nf);
        int r = job.fill(f0, nf, pin, src);
        if (r) return r;
        PMP_CUDA(cudaSetDevice(ln.h->device));
        for (int p = 0; p < nplanes; p++)
            PMP_CUDA(cudaMemcpyAsync(st.dev_in[s] + in_off(p, nf), src[p], (size_t)nf * rows[p] * prow[p],
                                     cudaMemcpyHostToDevice, st.copy));
        // cut and group on the copy stream, so that the distinct counts are on the host before compute(k) needs them
        const char *d = st.dev_in[s];
        r = cut_blocks(ln.h, d, chroma ? d + in_off(1, nf) : nullptr, chroma ? d + in_off(2, nf) : nullptr,
                       job.sample_bytes, nf, job.width, job.height, blocks_of(st, s, 0), blocks_of(st, s, 1), st.copy);
        if (r) return r;
        for (int c = 0; c < 2; c++)
            if (comp_on[c] && (r = group_blocks(ln.h, st.dev_group, st.group_cap, blocks_of(st, s, c), nf * bpf,
                                                (int)blk_bytes[c], 64, nullptr, groups_of(st.dev_group, st.group_cap, s, c),
                                                st.copy)))
                return r;
        PMP_CUDA(cudaMemcpyAsync(st.pin_count + 2 * s, groups_of(st.dev_group, st.group_cap, s, 0).count, 2 * sizeof(int),
                                 cudaMemcpyDeviceToHost, st.copy));
        PMP_CUDA(cudaEventRecord(st.uploaded[s], st.copy));
        return PMP_OK;
    };
    auto compute = [&](int k) -> int {
        Lane &ln = lanes[k % n];
        HostStage &st = *ln.st;
        pmp_handle *h = ln.h;
        const int j = k / n, s = j & 1, nf = win_frames(k);
        PMP_CUDA(cudaSetDevice(h->device));
        PMP_CUDA(cudaStreamWaitEvent(st.compute, st.uploaded[s], 0));
        if (j >= 2) PMP_CUDA(cudaStreamWaitEvent(st.compute, st.downloaded[s], 0));   // dev_out[s] read by j-2
        PMP_CUDA(cudaEventSynchronize(st.uploaded[s]));         // the distinct counts; in steady state long recorded
        char *o = st.dev_out[s];
        const long long N = (long long)nf * bpf;
        float *cqt = (float *)st.dev_work, *cbt = cqt + (size_t)chunk * 64, *cdi = cbt + (size_t)chunk * 768;
        uint8_t *qt8 = (uint8_t *)st.dev_work + maps_bytes, *compact = (uint8_t *)st.dev_work + off_compact,
                *qtx = (uint8_t *)st.dev_work + off_qtx, *expanded = (uint8_t *)st.dev_work + off_expanded;
        int r = PMP_OK;
        bool done[RESULTS_MAX] = {};
        for (int i = 0; i < nres; i++) {
            if (done[i]) continue;
            // the results that share result i's net pass: the same component and the same (Q, MSBD) weight sets
            const int c = res_c[i], wq = ln.wsets[4 * res_q[i] + 2 * c], wb = ln.wsets[4 * res_q[i] + 2 * c + 1];
            int grp[RESULTS_MAX], ng = 0;
            for (int j = i; j < nres; j++) {
                const int *wj = ln.wsets + 4 * res_q[j];
                if (!done[j] && res_c[j] == c && wj[2 * c] == wq && wj[2 * c + 1] == wb) {
                    grp[ng++] = j;
                    done[j] = true;
                }
            }
            auto dec = [&](int g) { return (uint8_t *)st.dev_work + off_rows + (size_t)g * row_bytes; };
            auto dec_flags = [&](int g) { return (uint32_t *)(dec(g) + dec_bytes); };
            // the net pass runs on the nd distinct blocks: in place without repeats, else gathered into compact order
            const Groups grps = groups_of(st.dev_group, st.group_cap, s, c);
            const int nd = st.pin_count[2 * s + c];
            const bool reuse = nd < N;
            const uint8_t *src = blocks_of(st, s, c);
            if (reuse) {
                if ((r = gather_blocks(h, src, grps.distinct, nd, (int)blk_bytes[c], compact, st.compute))) return r;
                src = compact;
            }
            st.stat_blocks += N;
            st.stat_computed += nd;
            for (long long b0 = 0; b0 < nd; b0 += chunk) {
                const int nb = (int)std::min<long long>(chunk, nd - b0);
                if ((r = pmp_predict_maps(h, wq, wb, src + b0 * blk_bytes[c], PMP_IN_U8, nb, cqt, cbt, cdi, st.compute)))
                    return r;
                if ((r = pmp_qt_postprocess(h, cqt, nb, nullptr, qt8 + b0 * 64, st.compute))) return r;
                for (int g = 0; g < ng; g++) {
                    const int k = grp[g];
                    uint8_t *d = dec(g);
                    r = pmp_map2partition_ex(h, qt8 + b0 * 64, cbt, cdi, nb, c == 0 ? 1 : 2,
                                             job.lamb ? job.lamb + 5 * res_q[k] : nullptr, cqt, h->near_tol,
                                             d + b0 * 256, d + (size_t)nmax * 256 + b0 * 256,
                                             (int8_t *)(d + (size_t)nmax * 512 + b0 * 768),
                                             (reuse ? dec_flags(g) : (uint32_t *)(o + off_flags[k])) + b0, st.compute);
                    if (r) return r;
                }
            }
            for (int g = 0; g < ng; g++) {
                const int k = grp[g];
                uint8_t *d = dec(g);
                if (reuse) {        // this row's maps and flags (and once the qt map) back to block order
                    r = expand_blocks(h, grps.slot, (int)N, nmax, d, expanded, dec_flags(g), (uint32_t *)(o + off_flags[k]),
                                      g == 0 ? qt8 : nullptr, qtx, st.compute);
                    if (r) return r;
                    d = expanded;
                }
                r = pmp_assemble_frames(h, d, d + (size_t)nmax * 256, reuse ? qtx : qt8,
                                        (const int8_t *)(d + (size_t)nmax * 512), nf, bh, bw, (int8_t *)(o + off_vals[k]),
                                        st.compute);
                if (r) return r;
                PMP_CUDA(cudaEventRecord(st.computed[s][k], st.compute));
            }
        }
        if (job.text) {
            const int8_t *vals[RESULTS_MAX];
            int64_t nv[RESULTS_MAX];
            char *txt[RESULTS_MAX];
            for (int i = 0; i < nres; i++) {
                vals[i] = (const int8_t *)(o + off_vals[i]);
                nv[i] = (int64_t)nf * per;
                txt[i] = o + off_text[i];
            }
            if ((r = format_texts(h, nres, vals, nv, txt, (int64_t *)(o + off_nbytes), st.compute))) return r;
        }
        PMP_CUDA(cudaMemcpyAsync(o + off_sat, h->d_status, sizeof(unsigned int), cudaMemcpyDeviceToDevice, st.compute));
        PMP_CUDA(cudaEventRecord(st.finished[s], st.compute));
        return PMP_OK;
    };
    auto download = [&](int k) -> int {        // a result's values leave while the next result's kernels run
        Lane &ln = lanes[k % n];
        HostStage &st = *ln.st;
        const int s = (k / n) & 1, f0 = k * wf, nf = win_frames(k);
        const char *o = st.dev_out[s];
        char *p = st.pin_out[s];
        PMP_CUDA(cudaSetDevice(ln.h->device));
        for (int i = 0; i < nres; i++) {
            PMP_CUDA(cudaStreamWaitEvent(st.copy, st.computed[s][i], 0));
            if (job.values) {
                int8_t *dst = direct(f0, i);
                PMP_CUDA(cudaMemcpyAsync(dst ? (char *)dst : p + off_vals[i], o + off_vals[i], (size_t)nf * per,
                                         cudaMemcpyDeviceToHost, st.copy));
            }
            PMP_CUDA(cudaMemcpyAsync(p + off_flags[i], o + off_flags[i], (size_t)nf * bpf * 4, cudaMemcpyDeviceToHost,
                                     st.copy));
        }
        PMP_CUDA(cudaStreamWaitEvent(st.copy, st.finished[s], 0));
        for (int i = 0; job.text && i < nres; i++)      // the byte counts are not known yet: the whole capacity
            PMP_CUDA(cudaMemcpyAsync(p + off_text[i], o + off_text[i], (size_t)3 * nf * per, cudaMemcpyDeviceToHost,
                                     st.copy));
        PMP_CUDA(cudaMemcpyAsync(p + off_nbytes, o + off_nbytes, off_sat + sizeof(unsigned int) - off_nbytes,
                                 cudaMemcpyDeviceToHost, st.copy));
        PMP_CUDA(cudaEventRecord(st.downloaded[s], st.copy));
        return PMP_OK;
    };
    auto finish = [&](int k) -> int {
        Lane &ln = lanes[k % n];
        HostStage &st = *ln.st;
        const int s = (k / n) & 1, f0 = k * wf, nf = win_frames(k);
        PMP_CUDA(cudaSetDevice(ln.h->device));
        PMP_CUDA(cudaEventSynchronize(st.downloaded[s]));
        const char *p = st.pin_out[s];
        pmp_window w;
        memset(&w, 0, sizeof(w));
        w.first_frame = f0;
        w.frames = nf;
        w.n_qps = job.n_qps;
        for (int i = 0; i < nres; i++) {
            const int q = res_q[i], c = res_c[i];
            w.n_values[q][c] = (int64_t)nf * per;
            if (job.values) {
                int8_t *dst = direct(f0, i);
                w.values[q][c] = dst ? dst : (const int8_t *)(p + off_vals[i]);
            }
            if (job.text) {
                w.text[q][c] = p + off_text[i];
                memcpy(&w.text_bytes[q][c], p + off_nbytes + 8 * i, 8);
            }
            const uint32_t *fl = (const uint32_t *)(p + off_flags[i]);
            for (long long b = 0; b < (long long)nf * bpf; b++) {      // the flag groups of ops.flag_counts
                w.report.blocks++;
                w.report.near_tie_blocks += (fl[b] & 1u) != 0;
                w.report.near_threshold_blocks += (fl[b] & 0xeu) != 0;
                w.report.near_threshold_blocks_tight += (fl[b] & 0x70u) != 0;
            }
        }
        unsigned int sat;
        memcpy(&sat, p + off_sat, sizeof(sat));
        w.report.fp16_saturation_events = (long long)(sat - ln.sat_prev);
        ln.sat_prev = sat;
        total->blocks += w.report.blocks;
        total->near_tie_blocks += w.report.near_tie_blocks;
        total->near_threshold_blocks += w.report.near_threshold_blocks;
        total->near_threshold_blocks_tight += w.report.near_threshold_blocks_tight;
        total->fp16_saturation_events += w.report.fp16_saturation_events;
        const int r = job.write(w);
        if (r) return r;
        if (job.stop_on_saturation && w.report.fp16_saturation_events) return saturation_error(total->fp16_saturation_events);
        return PMP_OK;
    };

    for (int k = 0; k < n && !rc; k++)
        if (!(rc = upload(k))) rc = compute(k);
    for (int k = 0; k < nwin && !rc; k++) {
        if (k >= n && (rc = compute(k))) break;
        if (k + n < nwin && (rc = upload(k + n))) break;
        if ((rc = download(k))) break;
        if (k >= n) rc = finish(k - n);
    }
    for (int k = std::max(0, nwin - n); k < nwin && !rc; k++) rc = finish(k);
    if (rc) {
        for (Lane &ln : lanes) {
            cudaSetDevice(ln.h->device);
            cudaStreamSynchronize(ln.st->compute);
            cudaStreamSynchronize(ln.st->copy);
        }
        return rc;
    }
    return total->fp16_saturation_events ? saturation_error(total->fp16_saturation_events) : PMP_OK;
}

// pmp_predict_stream over `n` handles: wsets [n][n_qps][4], lamb [n_qps][5] (checked by the caller) or nullptr, window
// k on hs[k % n].  caller >= 0 (the calling thread's device): pmp_predict_stream_multi's messages, which name the handle,
// and its device rule, `caller` current in every callback; -1: pmp_predict_stream's.
int predict_stream(pmp_handle *const *hs, int n, int n_qps, const int *wsets, const double *lamb, int frames, int width,
                   int height, int sample_bytes, int window_frames, int outputs, pmp_read_cb read, pmp_write_cb write,
                   void *user, pmp_report *report, int caller)
{
    const bool multi = caller >= 0;
    if (report) memset(report, 0, sizeof(*report));
    PMP_CHECK_ARG(n_qps >= 1 && n_qps <= 4, "n_qps must be 1 to 4");
    PMP_CHECK_ARG(wsets != nullptr, "null wsets");
    PMP_CHECK_ARG(read && write, "null callback");
    PMP_CHECK_ARG(outputs != 0 && (outputs & ~(PMP_OUT_VALUES | PMP_OUT_TEXT)) == 0,
                  "outputs must be PMP_OUT_VALUES, PMP_OUT_TEXT or both");
    PMP_CHECK_ARG(frames >= 0 && width >= 0 && height >= 0, "negative size");
    PMP_CHECK_ARG((width % 2) == 0 && (height % 2) == 0, "4:2:0 planes need even width and height");
    PMP_CHECK_ARG(sample_bytes == 1 || sample_bytes == 2, "sample_bytes must be 1 or 2");
    WindowJob job;
    bool chroma = false;
    for (int q = 0; q < n_qps; q++) {
        int rc = check_wsets(hs[0], wsets + 4 * q, 4 * q, job.on[q]);
        if (rc) {
            if (multi) set_error("handles[0]: %s", std::string(pmp_last_error()).c_str());
            return rc;
        }
        PMP_CHECK_ARG(job.on[q][0] || job.on[q][1], "both components of a QP are skipped");
        chroma = chroma || job.on[q][1];
    }
    // every other handle must compute what hs[0] computes: the same skip pattern, net kinds and weights, engine and
    // tc_dtype, and near_tol (the decode flags of the report)
    for (int i = 1; i < n; i++) {
        const Handle *a = hs[0], *b = hs[i];
        const int *wa = wsets, *wb = wsets + 4 * n_qps * i;
        auto differs = [&](const std::string &what) {
            set_error("bad argument: handles[%d] does not compute what handles[0] computes: %s", i, what.c_str());
            return PMP_ERR_ARG;
        };
        for (int q = 0; q < n_qps; q++) {
            bool on[2];
            int rc = check_wsets(b, wb + 4 * q, 4 * n_qps * i + 4 * q, on);
            if (rc) {
                set_error("handles[%d]: %s", i, std::string(pmp_last_error()).c_str());
                return rc;
            }
            for (int c = 0; c < 2; c++)
                if (on[c] != job.on[q][c])
                    return differs(std::string(c ? "chroma" : "luma") + " of QP row " + std::to_string(q) + " is " +
                                   (on[c] ? "run" : "skipped") + " here and " + (on[c] ? "skipped" : "run") + " there");
            for (int k = 0; k < 4; k++) {
                if (!on[k / 2]) continue;
                uint64_t fa, fb;
                if ((rc = wset_fingerprint(hs[0], wa[4 * q + k], &fa)) || (rc = wset_fingerprint(hs[i], wb[4 * q + k], &fb)))
                    return rc;
                if (fa != fb) {
                    char m[160];
                    snprintf(m, sizeof m, "the weights of wsets[%d][%d][%d] = %d (fingerprint %016llx, handles[0]'s %016llx)",
                             i, q, k, wb[4 * q + k], (unsigned long long)fb, (unsigned long long)fa);
                    return differs(m);
                }
            }
        }
        if (b->engine != a->engine)
            return differs("engine " + std::to_string(b->engine) + ", handles[0]'s " + std::to_string(a->engine));
        if (b->tc_dtype != a->tc_dtype)
            return differs("tc_dtype " + std::to_string(b->tc_dtype) + ", handles[0]'s " + std::to_string(a->tc_dtype));
        if (b->near_tol != a->near_tol) {
            char m[96];
            snprintf(m, sizeof m, "near_tol %g, handles[0]'s %g", b->near_tol, a->near_tol);
            return differs(m);
        }
    }
    const int bh = height / 64, bw = width / 64, bpf = bh * bw;
    if (frames == 0 || bpf == 0) return PMP_OK;
    // the default window: 4800 blocks, but small enough that every handle gets one
    const int wf = std::min(frames, window_frames > 0 ? window_frames : std::max(1, std::min(4800 / bpf, (frames + n - 1) / n)));
    PMP_CHECK_ARG((long long)wf * bpf < (1LL << 30) && (long long)wf * pmp_frame_values(bh, bw) <= TEXT_MAX_VALUES,
                  "too many blocks per window");
    job.n_qps = n_qps;
    job.lamb = lamb;
    job.frames = frames;
    job.width = width;
    job.height = height;
    job.sample_bytes = sample_bytes;
    job.wf = wf;
    job.values = (outputs & PMP_OUT_VALUES) != 0;
    job.text = (outputs & PMP_OUT_TEXT) != 0;
    job.stop_on_saturation = true;
    job.fill = [&](int f0, int nf, char *const pin[3], const char **) -> int {
        if (multi) PMP_CUDA(cudaSetDevice(caller));
        const int r = read(user, f0, nf, pin[0], chroma ? pin[1] : nullptr, chroma ? pin[2] : nullptr);
        if (r == 0) return PMP_OK;
        set_error("the read callback returned %d for frames %d..%d", r, f0, f0 + nf - 1);
        return PMP_ERR_ABORTED;
    };
    job.write = [&](const pmp_window &w) -> int {
        if (multi) PMP_CUDA(cudaSetDevice(caller));
        const int r = write(user, &w);
        if (r == 0) return PMP_OK;
        set_error("the write callback returned %d for frames %d..%d", r, w.first_frame, w.first_frame + w.frames - 1);
        return PMP_ERR_ABORTED;
    };
    std::vector<Lane> lanes(n);
    for (int i = 0; i < n; i++) {
        lanes[i].h = hs[i];
        lanes[i].wsets = wsets + 4 * n_qps * i;
    }
    pmp_report tot;
    const int rc = run_windows(lanes, job, &tot);
    if (report) *report = tot;
    return rc;
}

// pmp_predict_stream_multi and pmp_predict_stream_ex: the handle list's checks, then predict_stream with the calling
// thread's device current in the callbacks and restored on return.
int predict_stream_handles(pmp_handle *const *handles, int n_handles, int n_rows, const int *wsets, const double *lamb,
                           int frames, int width, int height, int sample_bytes, int window_frames, int outputs,
                           pmp_read_cb read, pmp_write_cb write, void *user, pmp_report *report)
{
    PMP_CHECK_ARG(n_handles >= 1 && n_handles <= STREAM_HANDLES_MAX, "n_handles must be 1 to 16");
    PMP_CHECK_ARG(handles != nullptr, "null handles");
    for (int i = 0; i < n_handles; i++) {
        if (!handles[i]) { set_error("bad argument: handles[%d] is null", i); return PMP_ERR_ARG; }
        for (int j = 0; j < i; j++)
            if (handles[j] == handles[i]) {
                set_error("bad argument: handles[%d] is handles[%d]: every handle must be distinct", i, j);
                return PMP_ERR_ARG;
            }
    }
    int caller = 0;
    PMP_CUDA(cudaGetDevice(&caller));
    const int rc = predict_stream(handles, n_handles, n_rows, wsets, lamb, frames, width, height, sample_bytes,
                                  window_frames, outputs, read, write, user, report, caller);
    cudaSetDevice(caller);
    return rc;
}

}  // namespace
}  // namespace pmp

using namespace pmp;

#define H_CHECK(h)                                                   \
    do {                                                             \
        if (!(h)) { set_error("null handle"); return PMP_ERR_ARG; }  \
        cudaError_t _e = cudaSetDevice((h)->device);                 \
        if (_e != cudaSuccess) return cuda_fail(_e, "cudaSetDevice", __FILE__, __LINE__); \
    } while (0)

extern "C" {

void pmp_destroy(pmp_handle *h)
{
    if (!h) return;
    release_stage(h);
    release_fingerprints(h);
    release_text_status(h);
    pmp_destroy_core(h);
}

int pmp_weights_load(pmp_handle *h, const char *path, int *net_out, int *wset)
{
    H_CHECK(h);
    PMP_CHECK_ARG(path && wset, "null pointer");
    return weights_load(h, path, net_out, wset);
}

int pmp_predict_host(pmp_handle *h, const int wsets[4], const void *y, const void *u, const void *v, int sample_bytes,
                     int64_t pitch_y, int64_t pitch_c, int frames, int width, int height, int chunk, int8_t *luma_out,
                     int8_t *chroma_out, pmp_report *report)
{
    H_CHECK(h);
    if (report) memset(report, 0, sizeof(*report));
    PMP_CHECK_ARG(wsets != nullptr, "null wsets");
    PMP_CHECK_ARG(frames >= 0 && width >= 0 && height >= 0, "negative size");
    PMP_CHECK_ARG((width % 2) == 0 && (height % 2) == 0, "4:2:0 planes need even width and height");
    PMP_CHECK_ARG(sample_bytes == 1 || sample_bytes == 2, "sample_bytes must be 1 or 2");
    WindowJob job;
    bool *on = job.on[0];
    int rc = check_wsets(h, wsets, 0, on);
    if (rc) return rc;
    PMP_CHECK_ARG(on[0] || on[1], "both components are skipped");
    const int bh = height / 64, bw = width / 64, bpf = bh * bw;
    if (frames == 0 || bpf == 0) return PMP_OK;
    PMP_CHECK_ARG(y && (!on[1] || (u && v)), "null input plane");
    int8_t *outs[2] = {luma_out, chroma_out};
    PMP_CHECK_ARG((!on[0] || luma_out) && (!on[1] || chroma_out), "null output");
    const int64_t row_y = (int64_t)width * sample_bytes, row_c = row_y / 2;
    if (pitch_y == 0) pitch_y = row_y;
    if (pitch_c == 0) pitch_c = row_c;
    PMP_CHECK_ARG(pitch_y >= row_y && pitch_c >= row_c, "pitch smaller than a row");
    if (chunk <= 0) chunk = 4800;
    job.n_qps = 1;
    job.frames = frames;
    job.width = width;
    job.height = height;
    job.sample_bytes = sample_bytes;
    job.chunk = chunk;
    job.wf = std::min(frames, std::max(1, chunk / bpf));
    PMP_CHECK_ARG((long long)job.wf * bpf < (1LL << 30), "too many blocks per window");
    const int64_t per = pmp_frame_values(bh, bw);

    const char *planes[3] = {(const char *)y, (const char *)u, (const char *)v};
    const int64_t pitch[3] = {pitch_y, pitch_c, pitch_c};
    const size_t rows[3] = {(size_t)height, (size_t)height / 2, (size_t)height / 2};
    const size_t prow[3] = {(size_t)row_y, (size_t)row_c, (size_t)row_c};
    const int nplanes = on[1] ? 3 : 1;
    // dense page-locked planes / outputs are copied directly; everything else goes through the pinned staging
    bool direct_in = true;
    for (int p = 0; p < nplanes; p++) direct_in = direct_in && pitch[p] == (int64_t)prow[p] && host_pinned(planes[p]);
    bool direct_out[2];
    for (int c = 0; c < 2; c++) direct_out[c] = on[c] && host_pinned(outs[c]);
    job.direct_in = direct_in;
    job.fill = [&](int f0, int nf, char *const pin[3], const char *src[3]) -> int {
        for (int p = 0; p < nplanes; p++) {
            const char *from = planes[p] + (size_t)f0 * rows[p] * pitch[p];
            if (direct_in) src[p] = from;
            else if (pitch[p] == (int64_t)prow[p]) memcpy(pin[p], from, (size_t)nf * rows[p] * prow[p]);
            else
                for (size_t r = 0; r < (size_t)nf * rows[p]; r++) memcpy(pin[p] + r * prow[p], from + r * pitch[p], prow[p]);
        }
        return PMP_OK;
    };
    job.direct_out = [&](int f0, int, int c) -> int8_t * { return direct_out[c] ? outs[c] + (size_t)f0 * per : nullptr; };
    job.write = [&](const pmp_window &w) -> int {
        for (int c = 0; c < 2; c++)
            if (on[c] && !direct_out[c]) memcpy(outs[c] + (size_t)w.first_frame * per, w.values[0][c], (size_t)w.n_values[0][c]);
        return PMP_OK;
    };
    std::vector<Lane> lanes(1);
    lanes[0].h = h;
    lanes[0].wsets = wsets;
    pmp_report tot;
    rc = run_windows(lanes, job, &tot);
    if (report && (rc == PMP_OK || rc == PMP_ERR_STATE)) *report = tot;
    return rc;
}

int pmp_format_texts(pmp_handle *h, int m, const int8_t *const *values, const int64_t *n, char *const *text,
                     int64_t *n_bytes, void *stream)
{
    H_CHECK(h);
    PMP_CHECK_ARG(m >= 1 && m <= TEXTS_MAX, "m must be 1 to 8");
    PMP_CHECK_ARG(values && n && text && n_bytes, "null pointer");
    for (int i = 0; i < m; i++) {
        PMP_CHECK_ARG(n[i] >= 0 && n[i] <= TEXT_MAX_VALUES, "a vector length is negative or above 2^30");
        PMP_CHECK_ARG(n[i] == 0 || (values[i] && text[i]), "null vector");
    }
    return format_texts(h, m, values, n, text, n_bytes, (cudaStream_t)stream);
}

int pmp_predict_stream(pmp_handle *h, int n_qps, const int *wsets, int frames, int width, int height, int sample_bytes,
                       int window_frames, int outputs, pmp_read_cb read, pmp_write_cb write, void *user,
                       pmp_report *report)
{
    H_CHECK(h);
    return predict_stream(&h, 1, n_qps, wsets, nullptr, frames, width, height, sample_bytes, window_frames, outputs, read,
                          write, user, report, -1);
}

int pmp_predict_stream_multi(pmp_handle *const *handles, int n_handles, int n_qps, const int *wsets, int frames,
                             int width, int height, int sample_bytes, int window_frames, int outputs, pmp_read_cb read,
                             pmp_write_cb write, void *user, pmp_report *report)
{
    if (report) memset(report, 0, sizeof(*report));
    return predict_stream_handles(handles, n_handles, n_qps, wsets, nullptr, frames, width, height, sample_bytes,
                                  window_frames, outputs, read, write, user, report);
}

int pmp_predict_stream_ex(pmp_handle *const *handles, int n_handles, int n_rows, const int *wsets, const double *lamb,
                          int frames, int width, int height, int sample_bytes, int window_frames, int outputs,
                          pmp_read_cb read, pmp_write_cb write, void *user, pmp_report *report)
{
    if (report) memset(report, 0, sizeof(*report));
    PMP_CHECK_ARG(n_rows >= 1 && n_rows <= 4, "n_rows must be 1 to 4");
    for (int r = 0; lamb && r < n_rows; r++)
        for (int k = 0; k < 5; k++)
            if (!std::isfinite(lamb[5 * r + k])) {
                set_error("bad argument: lamb[%d][%d] (row %d's lamb%d) is %g: every threshold must be finite", r, k, r,
                          k + 1, lamb[5 * r + k]);
                return PMP_ERR_ARG;
            }
    return predict_stream_handles(handles, n_handles, n_rows, wsets, lamb, frames, width, height, sample_bytes,
                                  window_frames, outputs, read, write, user, report);
}

int pmp_block_stats(pmp_handle *h, long long *blocks, long long *computed, int reset)
{
    H_CHECK(h);
    PMP_CHECK_ARG(blocks && computed, "null pointer");
    HostStage &st = stage_of(h);
    *blocks = st.stat_blocks;
    *computed = st.stat_computed;
    if (reset) st.stat_blocks = st.stat_computed = 0;
    return PMP_OK;
}

int pmp_debug_block_groups(pmp_handle *h, const uint8_t *blocks, int n, int block_bytes, int hash_bits, int *rep,
                           int *n_distinct_host, void *stream)
{
    H_CHECK(h);
    if (n_distinct_host) *n_distinct_host = 0;
    PMP_CHECK_ARG(n >= 0 && n < (1 << 30), "n must be 0 to 2^30 - 1");
    PMP_CHECK_ARG(block_bytes > 0 && block_bytes % 4 == 0, "block_bytes must be a positive multiple of 4");
    PMP_CHECK_ARG(hash_bits >= 0 && hash_bits <= 64, "hash_bits must be 0 to 64");
    if (n == 0) return PMP_OK;
    PMP_CHECK_ARG(blocks && rep, "null pointer");
    PMP_CHECK_ARG(((uintptr_t)blocks & 3) == 0, "blocks must be 4-byte aligned");
    HostStage &st = stage_of(h);
    int rc = ensure_group(st, n);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const Groups g = groups_of(st.dev_group, st.group_cap, 0, 0);
    if ((rc = group_blocks(h, st.dev_group, st.group_cap, blocks, n, block_bytes, hash_bits, rep, g, s))) return rc;
    int nd = 0;
    PMP_CUDA(cudaMemcpyAsync(&nd, g.count, sizeof(int), cudaMemcpyDeviceToHost, s));
    PMP_CUDA(cudaStreamSynchronize(s));
    if (n_distinct_host) *n_distinct_host = nd;
    return PMP_OK;
}

}  // extern "C"
