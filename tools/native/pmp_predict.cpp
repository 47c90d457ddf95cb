// pmp_predict: PartitionMat files from a YUV sequence without Python (C++11; include/pmp_b200.h + libpmp_b200.so only).
//
//   pmp_predict --input SEQ.yuv --width W --height H --frames N [--bitDepth 8|10] [--ssRatio S] [--qps 22,27,32,37]
//               --modelDir DIR --outDir DIR [--binaryOut] [--device D] [--tcDtype fp16|bf16] [--chunk C] [--timing]
//               [--stream]
//
// The weights are the exported .pmpw files (python -m pmp_vvc_tip2023_b200.export_weights): <comp>_Q_<qp>.pmpw and
// <comp>_BD_<qp>.pmpw in --modelDir.  Frames are read as Inference_QBD.import_yuv420 reads them (every S-th frame, by
// seek); per QP one pmp_predict_host call computes both components.  Writes
// <outDir>/<input basename without .yuv>_<comp>_QP<qp>_PartitionMat.txt (one decimal integer and '\n' per value,
// Map2Partition.py:405-412) and, with --binaryOut, the .bin beside it (32-byte "PMPPART1" header + raw int8 values,
// tools/vtm_reader/pmp_partition_reader.h).  Without --binaryOut an existing .bin is deleted, so that the VTM-side reader
// cannot pick up a stale one.  Nothing is written when the fp16 range guard fired (exit status 1: rerun with
// --tcDtype bf16).
//
// --stream makes one pmp_predict_stream call for all QPs instead: frames are read window by window straight into the
// library's page-locked planes, the GPU formats the text, and each window's text (and .bin payload) is appended to
// <stem>.txt.part (.bin.part) while the next window computes; the .part files are renamed once the call succeeds and
// deleted otherwise, so existing files are left as they were.  Host memory is bounded by the window (--chunk blocks,
// default 4800), not by the sequence.  The files are the same as without --stream.
#include "pmp_b200.h"

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <sys/stat.h>
#include <vector>

namespace {

struct Args {
    std::string input, model_dir, out_dir;
    int width = 0, height = 0, frames = 0, bit_depth = 8, ss_ratio = 1, device = 0, chunk = 0;
    std::vector<int> qps{22, 27, 32, 37};
    bool binary_out = false, bf16 = false, timing = false, stream = false;
};

int usage(const char *msg)
{
    std::fprintf(stderr,
                 "pmp_predict: %s\nusage: pmp_predict --input SEQ.yuv --width W --height H --frames N [--bitDepth 8|10] "
                 "[--ssRatio S] [--qps 22,27,32,37] --modelDir DIR --outDir DIR [--binaryOut] [--device D] "
                 "[--tcDtype fp16|bf16] [--chunk C] [--timing] [--stream]\n",
                 msg);
    return 2;
}

bool parse(int argc, char **argv, Args &a, std::string &err)
{
    for (int i = 1; i < argc; i++) {
        const std::string k = argv[i];
        if (k == "--binaryOut") { a.binary_out = true; continue; }
        if (k == "--timing") { a.timing = true; continue; }
        if (k == "--stream") { a.stream = true; continue; }
        if (i + 1 >= argc) { err = "missing value for " + k; return false; }
        const std::string v = argv[++i];
        if (k == "--input") a.input = v;
        else if (k == "--modelDir") a.model_dir = v;
        else if (k == "--outDir") a.out_dir = v;
        else if (k == "--width") a.width = std::atoi(v.c_str());
        else if (k == "--height") a.height = std::atoi(v.c_str());
        else if (k == "--frames") a.frames = std::atoi(v.c_str());
        else if (k == "--bitDepth") a.bit_depth = std::atoi(v.c_str());
        else if (k == "--ssRatio") a.ss_ratio = std::atoi(v.c_str());
        else if (k == "--device") a.device = std::atoi(v.c_str());
        else if (k == "--chunk") a.chunk = std::atoi(v.c_str());
        else if (k == "--tcDtype") {
            if (v != "fp16" && v != "bf16") { err = "--tcDtype must be fp16 or bf16"; return false; }
            a.bf16 = v == "bf16";
        } else if (k == "--qps") {
            a.qps.clear();
            for (size_t p = 0; p <= v.size();) {
                size_t q = v.find(',', p);
                if (q == std::string::npos) q = v.size();
                const int qp = std::atoi(v.substr(p, q - p).c_str());
                if (qp != 22 && qp != 27 && qp != 32 && qp != 37) { err = "QPs are 22, 27, 32, 37"; return false; }
                a.qps.push_back(qp);
                p = q + 1;
            }
        } else {
            err = "unknown option " + k;
            return false;
        }
    }
    if (a.input.empty() || a.model_dir.empty() || a.out_dir.empty()) { err = "--input, --modelDir and --outDir are required"; return false; }
    if (a.width <= 0 || a.height <= 0 || a.frames <= 0 || a.width % 2 || a.height % 2) { err = "bad --width/--height/--frames"; return false; }
    if (a.bit_depth != 8 && a.bit_depth != 10) { err = "--bitDepth must be 8 or 10"; return false; }
    if (a.ss_ratio < 1) { err = "--ssRatio must be at least 1"; return false; }
    return true;
}

// Inference_QBD.import_yuv420: frames 0, S, 2S, ... < N, each found by seeking; planes stored y[F] | u[F] | v[F].
bool read_yuv(const Args &a, int sb, std::vector<char> &buf, int &nf)
{
    const size_t pix = (size_t)a.width * a.height, ysz = pix * sb, csz = pix / 4 * sb;
    nf = (a.frames + a.ss_ratio - 1) / a.ss_ratio;
    buf.assign((size_t)nf * (ysz + 2 * csz), 0);
    FILE *fp = std::fopen(a.input.c_str(), "rb");
    if (!fp) { std::fprintf(stderr, "pmp_predict: cannot open %s\n", a.input.c_str()); return false; }
    char *y = buf.data(), *u = y + (size_t)nf * ysz, *v = u + (size_t)nf * csz;
    bool ok = true;
    for (int k = 0; k < nf && ok; k++) {
        const long long off = (long long)k * a.ss_ratio * (long long)(ysz + 2 * csz);
        ok = fseeko(fp, (off_t)off, SEEK_SET) == 0 && std::fread(y + k * ysz, 1, ysz, fp) == ysz &&
             std::fread(u + k * csz, 1, csz, fp) == csz && std::fread(v + k * csz, 1, csz, fp) == csz;
    }
    std::fclose(fp);
    if (!ok) std::fprintf(stderr, "pmp_predict: %s holds fewer than %d frames of %dx%d\n", a.input.c_str(), a.frames, a.width, a.height);
    return ok;
}

bool write_file(const std::string &path, const void *head, size_t head_n, const void *data, size_t n)
{
    FILE *fp = std::fopen(path.c_str(), "wb");
    bool ok = fp && (!head_n || std::fwrite(head, 1, head_n, fp) == head_n) && std::fwrite(data, 1, n, fp) == n;
    if (fp && std::fclose(fp) != 0) ok = false;
    if (!ok) std::fprintf(stderr, "pmp_predict: cannot write %s\n", path.c_str());
    return ok;
}

// Map2Partition.py:405-412: str(v) + '\n' per value, v in {-1, 0, 1, 2, 3}
bool write_text(const std::string &path, const std::vector<int8_t> &vals)
{
    static const char *const kText[5] = {"-1\n", "0\n", "1\n", "2\n", "3\n"};
    std::vector<char> txt;
    txt.reserve(vals.size() * 2 + vals.size() / 8);
    for (int8_t x : vals) {
        if (x < -1 || x > 3) { std::fprintf(stderr, "pmp_predict: value %d out of range\n", (int)x); return false; }
        const char *t = kText[x + 1];
        txt.insert(txt.end(), t, t + std::strlen(t));
    }
    return write_file(path, nullptr, 0, txt.data(), txt.size());
}

int fail(const char *what)
{
    std::fprintf(stderr, "pmp_predict: %s: %s\n", what, pmp_last_error());
    return 1;
}

void print_report(const pmp_report &tot)
{
    const double near_tol = 1e-2;      // the library's default (pmp_set_near_tol)
    std::printf("Decode report: %lld block-QPs, %lld float32 near-tie argmins, %lld with a map value within %g of a decision "
                "threshold (%lld within %g), %lld fp16 saturation events\n",
                tot.blocks, tot.near_tie_blocks, tot.near_threshold_blocks, near_tol, tot.near_threshold_blocks_tight,
                0.01 * near_tol, tot.fp16_saturation_events);
}

int saturated_exit(long long events)
{
    std::fprintf(stderr, "pmp_predict: activations left the fp16 range (%lld events): results are clamped; rerun with "
                         "--tcDtype bf16\n", events);
    return 1;
}

std::string stem_of(const Args &a, const std::string &base, int qp, int c)
{
    static const char *const comps[2] = {"Luma", "Chroma"};
    return a.out_dir + "/" + base + "_" + comps[c] + "_QP" + std::to_string(qp) + "_PartitionMat";
}

// ---- --stream ------------------------------------------------------------------------------------------------------
struct Stream {
    const Args *a;
    FILE *in = nullptr;
    size_t ysz = 0, csz = 0;
    int sb = 1;
    std::vector<FILE *> txt, bin;      // [2 * qp index + component]
    std::string io_error;
};

// Inference_QBD.import_yuv420's frames [f0, f0 + nf) of the subsampled sequence, into the library's planes
int stream_read(void *user, int f0, int nf, void *y, void *u, void *v)
{
    Stream &st = *static_cast<Stream *>(user);
    const Args &a = *st.a;
    for (int k = 0; k < nf; k++) {
        const long long off = (long long)(f0 + k) * a.ss_ratio * (long long)(st.ysz + 2 * st.csz);
        bool ok = fseeko(st.in, (off_t)off, SEEK_SET) == 0 && std::fread((char *)y + k * st.ysz, 1, st.ysz, st.in) == st.ysz;
        if (ok && u)
            ok = std::fread((char *)u + k * st.csz, 1, st.csz, st.in) == st.csz &&
                 std::fread((char *)v + k * st.csz, 1, st.csz, st.in) == st.csz;
        if (!ok) {
            st.io_error = a.input + " holds fewer than " + std::to_string(a.frames) + " frames of " + std::to_string(a.width) +
                          "x" + std::to_string(a.height);
            return 1;
        }
    }
    return 0;
}

int stream_write(void *user, const pmp_window *w)
{
    Stream &st = *static_cast<Stream *>(user);
    for (int q = 0; q < w->n_qps; q++)
        for (int c = 0; c < 2; c++) {
            const size_t i = 2 * q + c, nt = (size_t)w->text_bytes[q][c], nv = (size_t)w->n_values[q][c];
            if (std::fwrite(w->text[q][c], 1, nt, st.txt[i]) != nt || (st.bin[i] && std::fwrite(w->values[q][c], 1, nv, st.bin[i]) != nv)) {
                st.io_error = "write error";
                return 1;
            }
        }
    return 0;
}

int run_stream(const Args &a, pmp_handle *h, const std::vector<int> &wsets, const std::string &base)
{
    Stream st;
    st.a = &a;
    st.sb = a.bit_depth == 10 ? 2 : 1;
    st.ysz = (size_t)a.width * a.height * st.sb;
    st.csz = st.ysz / 4;
    const int nf = (a.frames + a.ss_ratio - 1) / a.ss_ratio, bh = a.height / 64, bw = a.width / 64, bpf = bh * bw;
    st.in = std::fopen(a.input.c_str(), "rb");
    if (!st.in) { std::fprintf(stderr, "pmp_predict: cannot open %s\n", a.input.c_str()); return 1; }
    mkdir(a.out_dir.c_str(), 0777);      // an existing directory is fine; a failure shows when the files are opened
    std::vector<std::string> parts;
    bool ok = true;
    for (size_t q = 0; q < a.qps.size() && ok; q++)
        for (int c = 0; c < 2 && ok; c++) {
            const std::string stem = stem_of(a, base, a.qps[q], c);
            parts.push_back(stem + ".txt.part");
            FILE *t = std::fopen(parts.back().c_str(), "wb");
            FILE *b = nullptr;
            if (t && a.binary_out) {
                parts.push_back(stem + ".bin.part");
                b = std::fopen(parts.back().c_str(), "wb");
                int32_t head32[8] = {0, 0, nf, 16 * bh, 16 * bw, 0, 0, 0};      // PMPPART1, frames, R, C, reserved
                std::memcpy(head32, "PMPPART1", 8);
                ok = b && std::fwrite(head32, 1, sizeof head32, b) == sizeof head32;
            }
            ok = ok && t;
            st.txt.push_back(t);
            st.bin.push_back(b);
            if (!ok) std::fprintf(stderr, "pmp_predict: cannot write %s\n", parts.back().c_str());
        }
    int rc = PMP_OK;
    pmp_report tot = {0, 0, 0, 0, 0};
    if (ok) {
        const auto t0 = std::chrono::steady_clock::now();
        const int window = a.chunk > 0 && bpf > 0 ? std::max(1, a.chunk / bpf) : 0;
        rc = pmp_predict_stream(h, (int)a.qps.size(), wsets.data(), nf, a.width, a.height, st.sb, window,
                                PMP_OUT_TEXT | (a.binary_out ? PMP_OUT_VALUES : 0), stream_read, stream_write, &st, &tot);
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        const int wf = window > 0 ? window : std::max(1, bpf > 0 ? 4800 / bpf : 1);
        if (a.timing) std::printf("pmp_predict_stream %.3f ms (%d frames, %d windows)\n", ms, nf, bpf > 0 ? (nf + wf - 1) / wf : 0);
    }
    std::fclose(st.in);
    for (size_t i = 0; i < st.txt.size(); i++) {
        if (st.txt[i] && std::fclose(st.txt[i]) != 0) st.io_error = "write error";
        if (st.bin[i] && std::fclose(st.bin[i]) != 0) st.io_error = "write error";
    }
    ok = ok && rc == PMP_OK && st.io_error.empty();
    if (ok) print_report(tot);
    for (size_t q = 0; q < a.qps.size() && ok; q++)
        for (int c = 0; c < 2 && ok; c++) {
            const std::string stem = stem_of(a, base, a.qps[q], c);
            ok = std::rename((stem + ".txt.part").c_str(), (stem + ".txt").c_str()) == 0;
            if (ok && a.binary_out) ok = std::rename((stem + ".bin.part").c_str(), (stem + ".bin").c_str()) == 0;
            else if (ok) std::remove((stem + ".bin").c_str());
            if (ok) std::printf("Save: %s.txt\n", stem.c_str());
            else std::fprintf(stderr, "pmp_predict: cannot rename %s.*.part\n", stem.c_str());
        }
    if (ok) return 0;
    for (const std::string &p : parts) std::remove(p.c_str());
    if (rc == PMP_ERR_STATE && tot.fp16_saturation_events) {
        print_report(tot);
        std::fprintf(stderr, "pmp_predict: %s\n", pmp_last_error());
        return saturated_exit(tot.fp16_saturation_events);
    }
    if (!st.io_error.empty()) std::fprintf(stderr, "pmp_predict: %s\n", st.io_error.c_str());
    if (rc != PMP_OK) return fail("pmp_predict_stream");
    return 1;
}

}  // namespace

int main(int argc, char **argv)
{
    Args a;
    std::string err;
    if (!parse(argc, argv, a, err)) return usage(err.c_str());
    pmp_handle *h = nullptr;
    if (pmp_create(a.device, &h) != PMP_OK) return fail("pmp_create");
    int rc = pmp_set_engine(h, PMP_ENGINE_TC, a.bf16 ? PMP_TC_BF16 : PMP_TC_FP16);
    if (rc) return fail("pmp_set_engine");

    const char *const comps[2] = {"Luma", "Chroma"};
    std::vector<int> wsets(4 * a.qps.size());
    for (size_t q = 0; q < a.qps.size(); q++)
        for (int c = 0; c < 2; c++)
            for (int k = 0; k < 2; k++) {
                const std::string path = a.model_dir + "/" + comps[c] + (k ? "_BD_" : "_Q_") + std::to_string(a.qps[q]) + ".pmpw";
                int net = -1;
                if (pmp_weights_load(h, path.c_str(), &net, &wsets[4 * q + 2 * c + k]) != PMP_OK) return fail("pmp_weights_load");
                if (net != 2 * c + k) {
                    std::fprintf(stderr, "pmp_predict: %s holds net kind %d, expected %d\n", path.c_str(), net, 2 * c + k);
                    return 1;
                }
            }

    std::string base = a.input.substr(a.input.find_last_of('/') + 1);
    if (base.size() > 4 && base.compare(base.size() - 4, 4, ".yuv") == 0) base.resize(base.size() - 4);
    if (a.stream) {
        rc = run_stream(a, h, wsets, base);
        pmp_destroy(h);
        return rc;
    }

    const int sb = a.bit_depth == 10 ? 2 : 1;
    std::vector<char> yuv;
    int nf = 0;
    if (!read_yuv(a, sb, yuv, nf)) return 1;
    const char *y = yuv.data(), *u = y + (size_t)nf * a.width * a.height * sb, *v = u + (size_t)nf * a.width * a.height / 4 * sb;
    const int bh = a.height / 64, bw = a.width / 64;
    const size_t n = (size_t)nf * (size_t)pmp_frame_values(bh, bw);

    // all QPs first: as in the Python driver, a saturating QP leaves no file behind
    std::vector<std::vector<int8_t> > out(2 * a.qps.size(), std::vector<int8_t>(n));
    pmp_report tot = {0, 0, 0, 0, 0};
    bool saturated = false;
    for (size_t q = 0; q < a.qps.size(); q++) {
        pmp_report r;
        const auto t0 = std::chrono::steady_clock::now();
        rc = pmp_predict_host(h, &wsets[4 * q], y, u, v, sb, 0, 0, nf, a.width, a.height, a.chunk, out[2 * q].data(),
                              out[2 * q + 1].data(), &r);
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (rc != PMP_OK && rc != PMP_ERR_STATE) return fail("pmp_predict_host");
        if (rc == PMP_ERR_STATE) {
            if (!r.fp16_saturation_events) return fail("pmp_predict_host");
            std::fprintf(stderr, "pmp_predict: QP %d: %s\n", a.qps[q], pmp_last_error());
            saturated = true;
        }
        if (a.timing) std::printf("QP %d: pmp_predict_host %.3f ms (%d frames, %d blocks per component)\n", a.qps[q], ms, nf, nf * bh * bw);
        tot.blocks += r.blocks;
        tot.near_tie_blocks += r.near_tie_blocks;
        tot.near_threshold_blocks += r.near_threshold_blocks;
        tot.near_threshold_blocks_tight += r.near_threshold_blocks_tight;
        tot.fp16_saturation_events += r.fp16_saturation_events;
    }
    pmp_destroy(h);
    print_report(tot);
    if (saturated) return saturated_exit(tot.fp16_saturation_events);

    mkdir(a.out_dir.c_str(), 0777);      // an existing directory is fine; a failure shows when the files are written
    for (size_t q = 0; q < a.qps.size(); q++)
        for (int c = 0; c < 2; c++) {
            const std::string stem = stem_of(a, base, a.qps[q], c);
            std::printf("Save: %s.txt\n", stem.c_str());
            if (!write_text(stem + ".txt", out[2 * q + c])) return 1;
            if (a.binary_out) {
                int32_t head32[8] = {0, 0, nf, 16 * bh, 16 * bw, 0, 0, 0};      // PMPPART1, frames, R, C, reserved
                std::memcpy(head32, "PMPPART1", 8);
                if (!write_file(stem + ".bin", head32, sizeof head32, out[2 * q + c].data(), n)) return 1;
            } else {
                std::remove((stem + ".bin").c_str());
            }
        }
    return 0;
}
