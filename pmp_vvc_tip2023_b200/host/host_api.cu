// Host-level entry points of libpmp_b200 for callers without Python or CUDA of their own (include/pmp_b200.h):
// pmp_weights_load (exported .pmpw weight files) and pmp_predict_host (host planes in, host PartitionMat vectors out),
// plus pmp_destroy, which releases this layer's staging before the core handle teardown in csrc/api.cu.
//
// This layer only calls the core's entry points and internal functions; it lives outside csrc/ because bench.py ties
// the committed ncu traffic summary (profiles/r*_traffic.json) to a hash of the csrc/ sources, and none of those kernels
// change here.  build.py compiles csrc/api.cu with -Dpmp_destroy=pmp_destroy_core so that the exported pmp_destroy is
// the one below.
#include "../csrc/handle.cuh"

#include <algorithm>
#include <cstdio>
#include <cstring>
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

uint64_t fnv1a64(const unsigned char *p, size_t n)
{
    uint64_t x = 0xcbf29ce484222325ull;
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

// ---- staging of pmp_predict_host ---------------------------------------------------------------------------------
// Per handle: a compute and a copy stream, their events, and per window slot (double-buffered) pinned + device buffers
// for the input planes and for the outputs (values and decode flags of both components).  Created on first use, grown
// to the largest window, released by pmp_destroy.
struct HostStage {
    cudaStream_t compute = nullptr, copy = nullptr;
    cudaEvent_t uploaded[2] = {}, cut[2] = {}, downloaded[2] = {}, computed[2][2] = {};
    char *pin_in[2] = {}, *pin_out[2] = {}, *dev_in[2] = {}, *dev_out[2] = {};
    uint8_t *dev_blocks = nullptr;
    size_t in_bytes = 0, out_bytes = 0, blocks_bytes = 0;     // per slot
};

std::mutex g_stage_mu;
std::map<const Handle *, HostStage> g_stage;     // a handle is used by one thread at a time; the map by all

HostStage &stage_of(const Handle *h)
{
    std::lock_guard<std::mutex> lock(g_stage_mu);
    return g_stage[h];
}

void free_buffers(HostStage &st)
{
    for (int s = 0; s < 2; s++) {
        if (st.pin_in[s]) cudaFreeHost(st.pin_in[s]);
        if (st.pin_out[s]) cudaFreeHost(st.pin_out[s]);
        if (st.dev_in[s]) cudaFree(st.dev_in[s]);
        if (st.dev_out[s]) cudaFree(st.dev_out[s]);
        st.pin_in[s] = st.pin_out[s] = st.dev_in[s] = st.dev_out[s] = nullptr;
    }
    if (st.dev_blocks) cudaFree(st.dev_blocks);
    st.dev_blocks = nullptr;
    st.in_bytes = st.out_bytes = st.blocks_bytes = 0;
}

int ensure_stage(HostStage &st, size_t in_bytes, size_t out_bytes, size_t blocks_bytes)
{
    if (!st.compute) {
        PMP_CUDA(cudaStreamCreateWithFlags(&st.compute, cudaStreamNonBlocking));
        PMP_CUDA(cudaStreamCreateWithFlags(&st.copy, cudaStreamNonBlocking));
        for (int s = 0; s < 2; s++)
            for (cudaEvent_t *e : {&st.uploaded[s], &st.cut[s], &st.downloaded[s], &st.computed[s][0], &st.computed[s][1]})
                PMP_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    }
    if (in_bytes <= st.in_bytes && out_bytes <= st.out_bytes && blocks_bytes <= st.blocks_bytes) return PMP_OK;
    in_bytes = std::max(in_bytes, st.in_bytes);
    out_bytes = std::max(out_bytes, st.out_bytes);
    blocks_bytes = std::max(blocks_bytes, st.blocks_bytes);
    free_buffers(st);       // the previous call ended synchronised: nothing in flight uses them
    for (int s = 0; s < 2; s++) {
        PMP_CUDA(cudaHostAlloc((void **)&st.pin_in[s], in_bytes, cudaHostAllocDefault));
        PMP_CUDA(cudaHostAlloc((void **)&st.pin_out[s], out_bytes, cudaHostAllocDefault));
        PMP_CUDA(cudaMalloc((void **)&st.dev_in[s], in_bytes));
        PMP_CUDA(cudaMalloc((void **)&st.dev_out[s], out_bytes));
    }
    PMP_CUDA(cudaMalloc((void **)&st.dev_blocks, blocks_bytes));
    st.in_bytes = in_bytes;
    st.out_bytes = out_bytes;
    st.blocks_bytes = blocks_bytes;
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
    for (int s = 0; s < 2; s++)
        for (cudaEvent_t e : {st.uploaded[s], st.cut[s], st.downloaded[s], st.computed[s][0], st.computed[s][1]})
            cudaEventDestroy(e);
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
    bool on[2];
    for (int c = 0; c < 2; c++) {
        on[c] = !(wsets[2 * c] == -1 && wsets[2 * c + 1] == -1);
        for (int k = 0; on[c] && k < 2; k++) {
            auto it = h->wsets.find(wsets[2 * c + k]);
            if (it == h->wsets.end() || it->second.net != 2 * c + k) {
                set_error("wsets[%d] = %d is not a weight set of net kind %d", 2 * c + k, wsets[2 * c + k], 2 * c + k);
                return PMP_ERR_ARG;
            }
        }
    }
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

    // windows of whole frames; per slot: dense planes in, values + decode flags of both components out
    const int wf = std::min(frames, std::max(1, chunk / bpf));
    const long long nmax = (long long)wf * bpf;
    PMP_CHECK_ARG(nmax < (1LL << 30), "too many blocks per window");
    const int64_t per = pmp_frame_values(bh, bw);
    const size_t plane_y = (size_t)height * row_y, plane_c = (size_t)(height / 2) * row_c;
    const size_t in_frame = plane_y + (on[1] ? 2 * plane_c : 0);
    const size_t vals_bytes = ((size_t)wf * per + 255) & ~(size_t)255, flags_bytes = ((size_t)nmax * 4 + 255) & ~(size_t)255;
    const size_t off_vals[2] = {0, vals_bytes}, off_flags[2] = {2 * vals_bytes, 2 * vals_bytes + flags_bytes};
    const size_t blk_bytes[2] = {(size_t)68 * 68, (size_t)3 * 34 * 34};
    HostStage &st = stage_of(h);
    int rc = ensure_stage(st, (size_t)wf * in_frame, 2 * vals_bytes + 2 * flags_bytes,
                          (size_t)nmax * ((on[0] ? blk_bytes[0] : 0) + (on[1] ? blk_bytes[1] : 0)));
    if (rc) return rc;
    // The status word exists before the loop (ensure_status allocates on the legacy stream).  The arena and scratch grow
    // inside the first window's pmp_run_component when a handle first sees this window size; that synchronises the
    // device once and leaves everything queued intact.
    if ((rc = ensure_status(h))) return rc;
    PMP_CUDA(cudaDeviceSynchronize());
    unsigned int sat0 = 0, sat1 = 0;
    PMP_CUDA(cudaMemcpy(&sat0, h->d_status, sizeof(sat0), cudaMemcpyDeviceToHost));

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
    const int nwin = (frames + wf - 1) / wf;
    auto win_frames = [&](int k) { return std::min(wf, frames - k * wf); };
    auto in_off = [&](int p, int nf) { return p == 0 ? 0 : (size_t)nf * (plane_y + (p - 1) * plane_c); };

    auto upload = [&](int k) -> int {
        const int s = k & 1, f0 = k * wf, nf = win_frames(k);
        if (k >= 2) {
            if (!direct_in) PMP_CUDA(cudaEventSynchronize(st.uploaded[s]));     // pin_in[s] free again
            PMP_CUDA(cudaStreamWaitEvent(st.copy, st.cut[s], 0));               // dev_in[s] read by window k-2's cut
        }
        for (int p = 0; p < nplanes; p++) {
            const char *src = planes[p] + (size_t)f0 * rows[p] * pitch[p];
            if (!direct_in) {
                char *dst = st.pin_in[s] + in_off(p, nf);
                if (pitch[p] == (int64_t)prow[p]) memcpy(dst, src, (size_t)nf * rows[p] * prow[p]);
                else
                    for (size_t r = 0; r < (size_t)nf * rows[p]; r++) memcpy(dst + r * prow[p], src + r * pitch[p], prow[p]);
                src = dst;
            }
            PMP_CUDA(cudaMemcpyAsync(st.dev_in[s] + in_off(p, nf), src, (size_t)nf * rows[p] * prow[p],
                                     cudaMemcpyHostToDevice, st.copy));
        }
        PMP_CUDA(cudaEventRecord(st.uploaded[s], st.copy));
        return PMP_OK;
    };
    auto compute = [&](int k) -> int {
        const int s = k & 1, nf = win_frames(k);
        PMP_CUDA(cudaStreamWaitEvent(st.compute, st.uploaded[s], 0));
        if (k >= 2) PMP_CUDA(cudaStreamWaitEvent(st.compute, st.downloaded[s], 0));   // dev_out[s] read by window k-2
        const char *d = st.dev_in[s];
        uint8_t *blk[2] = {on[0] ? st.dev_blocks : nullptr,
                           on[1] ? st.dev_blocks + (on[0] ? (size_t)nmax * blk_bytes[0] : 0) : nullptr};
        int r = cut_blocks(h, d, on[1] ? d + in_off(1, nf) : nullptr, on[1] ? d + in_off(2, nf) : nullptr, sample_bytes, nf,
                           width, height, blk[0], blk[1], st.compute);
        if (r) return r;
        PMP_CUDA(cudaEventRecord(st.cut[s], st.compute));
        for (int c = 0; c < 2; c++) {
            if (!on[c]) continue;
            r = pmp_run_component(h, wsets[2 * c], wsets[2 * c + 1], c == 0, blk[c], nf, bh, bw, chunk,
                                  (int8_t *)(st.dev_out[s] + off_vals[c]), nullptr, nullptr, nullptr,
                                  (uint32_t *)(st.dev_out[s] + off_flags[c]), st.compute);
            if (r) return r;
            PMP_CUDA(cudaEventRecord(st.computed[s][c], st.compute));
        }
        return PMP_OK;
    };
    auto download = [&](int k) -> int {        // luma's copy overlaps chroma's kernels
        const int s = k & 1, nf = win_frames(k);
        for (int c = 0; c < 2; c++) {
            if (!on[c]) continue;
            PMP_CUDA(cudaStreamWaitEvent(st.copy, st.computed[s][c], 0));
            PMP_CUDA(cudaMemcpyAsync(direct_out[c] ? (char *)(outs[c] + (size_t)k * wf * per) : st.pin_out[s] + off_vals[c],
                                     st.dev_out[s] + off_vals[c], (size_t)nf * per, cudaMemcpyDeviceToHost, st.copy));
            PMP_CUDA(cudaMemcpyAsync(st.pin_out[s] + off_flags[c], st.dev_out[s] + off_flags[c], (size_t)nf * bpf * 4,
                                     cudaMemcpyDeviceToHost, st.copy));
        }
        PMP_CUDA(cudaEventRecord(st.downloaded[s], st.copy));
        return PMP_OK;
    };
    long long counts[4] = {0, 0, 0, 0};
    auto finish = [&](int k) -> int {
        const int s = k & 1, nf = win_frames(k);
        PMP_CUDA(cudaEventSynchronize(st.downloaded[s]));
        for (int c = 0; c < 2; c++) {
            if (!on[c]) continue;
            if (!direct_out[c]) memcpy(outs[c] + (size_t)k * wf * per, st.pin_out[s] + off_vals[c], (size_t)nf * per);
            const uint32_t *fl = (const uint32_t *)(st.pin_out[s] + off_flags[c]);
            for (long long b = 0; b < (long long)nf * bpf; b++) {      // the flag groups of ops.flag_counts
                counts[0]++;
                counts[1] += (fl[b] & 1u) != 0;
                counts[2] += (fl[b] & 0xeu) != 0;
                counts[3] += (fl[b] & 0x70u) != 0;
            }
        }
        return PMP_OK;
    };

    // window k+1 uploads and window k-1 downloads while window k computes
    rc = upload(0);
    for (int k = 0; k < nwin && !rc; k++) {
        if (k + 1 < nwin && (rc = upload(k + 1))) break;
        if ((rc = compute(k)) || (rc = download(k))) break;
        if (k >= 1) rc = finish(k - 1);
    }
    if (!rc) rc = finish(nwin - 1);
    if (rc) {
        cudaStreamSynchronize(st.compute);
        cudaStreamSynchronize(st.copy);
        return rc;
    }
    PMP_CUDA(cudaMemcpy(&sat1, h->d_status, sizeof(sat1), cudaMemcpyDeviceToHost));
    const long long sat = (long long)(sat1 - sat0);
    if (report) {
        report->blocks = counts[0];
        report->near_tie_blocks = counts[1];
        report->near_threshold_blocks = counts[2];
        report->near_threshold_blocks_tight = counts[3];
        report->fp16_saturation_events = sat;
    }
    if (sat) {
        set_error("%lld fp16 saturation events: activations left the fp16 range and the results are clamped; rerun with "
                  "PMP_TC_BF16 (pmp_set_engine)", sat);
        return PMP_ERR_STATE;
    }
    return PMP_OK;
}

}  // extern "C"
