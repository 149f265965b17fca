// gpsb200-sim: file-sink driver with the reference's command-line vocabulary (help.h:20-53:
// -e nav file, -l location, -t target, -d duration, -m motion file, -s start, --iq16, -I no ionosphere) and
// --almanac FILE: the almanac pages the reference builds from its almanac.sem, from a local SEM file.
// RINEX + location -> scenario engine (host) -> CUDA synthesis -> reference-compatible FIFO ->
// iqfile writer. Output is byte-identical to the reference's enqueue stream; --compat-drop
// reproduces the stock program's iqdata.bin (which lacks blocks 1..6, fifo.c:163-168).
//
// One GPU: the FIFO is created with a batch worth of page-locked buffers; every batch is synthesized with
// gpsb200_synth_blocks_scatter, i.e. the device->host copies land straight in the acquired iq->data8/16 (no staging
// copy), and the buffers are enqueued in order.
// --gpus N: the stream is cut into N contiguous time slices, one worker thread and one context per device. The
// slices' closed-form links give every worker a guessed incoming carrier-chain state at once (gpsb200_slice_link_host
// + gpsb200_link_apply), all workers probe speculatively in parallel, and the exact states travel worker to worker
// (gpsb200_slice_prepare / _probe / _finish). Each worker downloads into a page-locked slice buffer; the main thread
// feeds the slices to the FIFO in stream order as they complete.
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime_api.h>

#include "../include/gpsb200.h"

static void usage() {
    fprintf(stderr,
            "gpsb200-sim -e NAV[.gz] [-3] -l lat,lon,h [-t dist,bearing,height] [-d SEC] [-m motion.csv] [-s y/m/d,h:m:s]\n"
            "            [--iq16] [-I] [--pluto-gain] [--chan N] [--gpus N] [-o iqdata.bin] [--compat-drop] [--u32-carrier]\n"
            "            [--almanac FILE]\n"
            "  --almanac FILE: SEM almanac for subframes 4/5 (the reference's almanac.sem; without it: no almanac pages)\n"
            "  --u32-carrier: the stream of the reference built without FLOAT_CARR_PHASE (gps.h:17): integer carrier NCO\n");
    exit(2);
}

static double now_s() {
    using namespace std::chrono;
    return duration<double>(steady_clock::now().time_since_epoch()).count();
}

namespace {
struct Handoff {                 // exact chain state after slice r, published by worker r
    std::mutex mu;
    std::condition_variable cv;
    bool ready = false, failed = false;
    std::vector<int32_t> prn;
    std::vector<double> phase;
};
}  // namespace

int main(int argc, char **argv) {
    gpsb200_scenario_config_t sc{};
    sc.ionosphere_enable = 1;
    sc.max_chan = 12;
    double dur = 300.0;
    int sample_size = GPSB200_SC08, gpus = 1, carrier = GPSB200_CARRIER_FP64;
    bool compat = false;
    std::string out = "iqdata.bin";
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        auto need = [&]() -> const char * {
            if (i + 1 >= argc) usage();
            return argv[++i];
        };
        if (a == "-e") sc.nav_file = need();
        else if (a == "-l") sscanf(need(), "%lf,%lf,%lf", &sc.lat_deg, &sc.lon_deg, &sc.height_m);
        else if (a == "-t") {
            sc.target_valid = 1;                                    // gps-sim.c:145-148
            sscanf(need(), "%lf,%lf,%lf", &sc.target_distance_m, &sc.target_bearing_deg, &sc.target_height_m);
        } else if (a == "-d") dur = atof(need());
        else if (a == "-m") sc.motion_file = need();
        else if (a == "-s")
            sscanf(need(), "%d/%d/%d,%d:%d:%lf", &sc.start_year, &sc.start_month, &sc.start_day, &sc.start_hour,
                   &sc.start_min, &sc.start_sec);
        else if (a == "--iq16") sample_size = GPSB200_SC16;
        else if (a == "-I") sc.ionosphere_enable = 0;
        else if (a == "-3") sc.rinex3 = 1;
        else if (a == "--pluto-gain") sc.pluto_gain = 1;
        else if (a == "--chan") sc.max_chan = atoi(need());
        else if (a == "--gpus") gpus = atoi(need());
        else if (a == "-o") out = need();
        else if (a == "--compat-drop") compat = true;
        else if (a == "--u32-carrier") carrier = GPSB200_CARRIER_U32;
        else if (a == "--almanac") sc.almanac_file = need();
        else usage();
    }
    if (!sc.nav_file || gpus < 1) usage();
    sc.duration_ds = (int) (dur * 10.0 + 0.5);                  // gps-sim.c:140
    sc.carrier_u32 = carrier == GPSB200_CARRIER_U32;            // allocation phases of that build (gps.c:2212-2213)

    gpsb200_scenario_t *scn = nullptr;
    if (gpsb200_scenario_create(&sc, &scn) != GPSB200_OK) {
        fprintf(stderr, "scenario: %s\n", gpsb200_scenario_error(scn));
        return 1;
    }
    const int nblk = gpsb200_scenario_blocks(scn), nchan = gpsb200_scenario_channels(scn);
    const int nframes = gpsb200_scenario_nav_frames(scn);
    if (!sc.almanac_file)
        fprintf(stderr, "gpsb200-sim: note: no almanac pages are generated -- the stream equals the reference's with its almanac "
                        "disabled (the reference enables it by default and downloads one); --almanac FILE adds them\n");
    const gpsb200_chan_t *chans = gpsb200_scenario_chans(scn);
    const uint32_t *nav = gpsb200_scenario_nav(scn);
    const size_t blk_bytes = (size_t) GPSB200_BLOCK_ELEMS * sample_size;
    int ndev = 0;
    cudaGetDeviceCount(&ndev);
    if (gpus > ndev) {
        fprintf(stderr, "gpsb200-sim: --gpus %d but %d CUDA device(s) visible\n", gpus, ndev);
        return 1;
    }
    gpus = std::min(gpus, std::max(1, nblk));
    const double t0 = now_s();

    auto make_ctx = [&](int dev, int max_blocks, gpsb200_ctx_t **ctx) -> bool {
        gpsb200_config_t cfg{};
        cfg.device = dev;
        cfg.max_chan = nchan;
        cfg.max_blocks = max_blocks;
        cfg.max_nav_frames = nframes;
        cfg.carrier_nco = carrier;
        if (gpsb200_create(&cfg, ctx) != GPSB200_OK) {
            fprintf(stderr, "gpsb200: %s\n", gpsb200_last_error(*ctx));
            return false;
        }
        for (int f = 0; f < nframes; f++)
            for (int c = 0; c < nchan; c++)
                gpsb200_set_nav(*ctx, f, c, nav + ((size_t) f * nchan + c) * GPSB200_NAV_WORDS);
        return true;
    };

    fifo_set_compat_drop(compat);
    bool writer = false;
    int queued = 0;
    auto start_writer_if_primed = [&](bool force) -> bool {
        // like the reference (sdr_iqfile.c:73-77) the writer starts once the FIFO is primed (or the run ends)
        if (!writer && (queued >= 8 || force)) {
            if (gpsb200_iqfile_start(out.c_str(), sample_size) != GPSB200_OK) return false;
            writer = true;
        }
        return true;
    };

    if (gpus == 1) {
        const int batch = std::min(256, nblk);
        gpsb200_ctx_t *ctx = nullptr;
        gpsb200_bind_numa(0);           // threads and pinned FIFO buffers next to the GPU (cf. thread_to_core, gps.c:2377)
        if (!make_ctx(0, batch, &ctx)) return 1;
        // a batch worth of FIFO buffers (+ the 8 the reference keeps in flight, sdr.h:24): every block of a batch is
        // downloaded straight into its own acquired buffer. --compat-drop reproduces a property of the reference's
        // 8-buffer FIFO, so it keeps that geometry and goes through a staging buffer.
        void *stage = nullptr;
        if (compat && cudaHostAlloc(&stage, blk_bytes * batch, cudaHostAllocDefault) != cudaSuccess) return 1;
        if (!fifo_create(compat ? 8u : (unsigned) batch + 8, GPSB200_BLOCK_ELEMS, sample_size)) return 1;
        std::vector<double> carr(nchan, 0.0);
        std::vector<gpsb200_chan_t> part;
        std::vector<struct iq_buf *> bufs;
        std::vector<void *> dsts;
        for (int b0 = 0; b0 < nblk; b0 += batch) {
            const int nb = std::min(batch, nblk - b0);
            part.assign(chans + (size_t) b0 * nchan, chans + (size_t) (b0 + nb) * nchan);
            if (b0 > 0)                                             // continue the carrier chain across calls
                for (int c = 0; c < nchan; c++)
                    if (part[c].prn > 0 && part[c].prn == chans[(size_t) (b0 - 1) * nchan + c].prn) part[c].carr_phase = carr[c];
            if (compat) {
                if (gpsb200_synth_blocks(ctx, part.data(), nb, nchan, sample_size, stage, carr.data(), nullptr) != GPSB200_OK) {
                    fprintf(stderr, "gpsb200: %s\n", gpsb200_last_error(ctx));
                    return 1;
                }
                for (int b = 0; b < nb; b++) {
                    if (!start_writer_if_primed(false)) return 1;
                    struct iq_buf *iq = fifo_acquire();
                    if (!iq) return 1;
                    memcpy(sample_size == GPSB200_SC16 ? (void *) iq->data16 : (void *) iq->data8,
                           (char *) stage + (size_t) b * blk_bytes, blk_bytes);
                    iq->validLength = GPSB200_BLOCK_ELEMS;
                    fifo_enqueue(iq);
                    queued++;
                }
                continue;
            }
            bufs.assign(nb, nullptr);
            dsts.assign(nb, nullptr);
            for (int b = 0; b < nb; b++) {
                bufs[b] = fifo_acquire();                           // gps.c:2698 / 2864
                if (!bufs[b]) return 1;
                dsts[b] = sample_size == GPSB200_SC16 ? (void *) bufs[b]->data16 : (void *) bufs[b]->data8;
            }
            if (gpsb200_synth_blocks_scatter(ctx, part.data(), nb, nchan, sample_size, dsts.data(), carr.data(), nullptr) !=
                GPSB200_OK) {
                fprintf(stderr, "gpsb200: %s\n", gpsb200_last_error(ctx));
                return 1;
            }
            for (int b = 0; b < nb; b++) {
                if (!start_writer_if_primed(false)) return 1;
                bufs[b]->validLength = GPSB200_BLOCK_ELEMS;
                fifo_enqueue(bufs[b]);                              // gps.c:2860
                queued++;
            }
        }
        if (!start_writer_if_primed(true)) return 1;
        gpsb200_iqfile_stop();
        fifo_destroy();
        if (stage) cudaFreeHost(stage);
        gpsb200_destroy(ctx);
    } else {
        // ---- time slices over several GPUs ----------------------------------------------------------------
        std::vector<int> lo(gpus + 1, 0);
        for (int r = 0; r < gpus; r++) {
            const int base = nblk / gpus, extra = nblk % gpus;
            lo[r + 1] = lo[r] + base + (r < extra ? 1 : 0);
        }
        // guessed incoming states from the closed-form links (exact with --u32-carrier): no GPU work, no dependence between
        // the workers
        std::vector<std::vector<int32_t>> gprn(gpus, std::vector<int32_t>(nchan, 0));
        std::vector<std::vector<double>> gph(gpus, std::vector<double>(nchan, 0.0));
        {
            std::vector<int32_t> p(nchan, 0), pn(nchan, 0);
            std::vector<double> x(nchan, 0.0), xn(nchan, 0.0);
            bool have = false;
            for (int r = 0; r < gpus; r++) {
                gprn[r] = p;
                gph[r] = x;
                gpsb200_slice_link_t link;
                if (gpsb200_slice_link_host_nco(chans + (size_t) lo[r] * nchan, lo[r + 1] - lo[r], nchan, carrier, &link) !=
                    GPSB200_OK)
                    return 1;
                gpsb200_link_apply_nco(&link, nchan, carrier, have ? p.data() : nullptr, have ? x.data() : nullptr, pn.data(),
                                       xn.data());
                p = pn;
                x = xn;
                have = true;
            }
        }
        std::vector<Handoff> hand(gpus);
        std::vector<void *> slice_host(gpus, nullptr);
        std::vector<int> done(gpus, 0);            // 0 running, 1 ok, -1 failed
        std::mutex done_mu;
        std::condition_variable done_cv;
        std::vector<std::thread> workers;
        for (int r = 0; r < gpus; r++) {
            workers.emplace_back([&, r] {
                const int nb = lo[r + 1] - lo[r];
                bool ok = false;
                gpsb200_ctx_t *ctx = nullptr;
                std::vector<int32_t> prn_out(nchan, 0);
                std::vector<double> ph_out(nchan, 0.0);
                do {
                    if (cudaSetDevice(r) != cudaSuccess) break;
                    gpsb200_bind_numa(r);
                    if (cudaHostAlloc(&slice_host[r], blk_bytes * nb, cudaHostAllocPortable) != cudaSuccess) break;
                    if (!make_ctx(r, nb, &ctx)) break;
                    gpsb200_slice_link_t link;
                    if (gpsb200_slice_prepare(ctx, chans + (size_t) lo[r] * nchan, nb, nchan, sample_size, nullptr, slice_host[r],
                                              nullptr, &link) != GPSB200_OK) break;
                    if (gpsb200_slice_probe(ctx, r ? gprn[r].data() : nullptr, r ? gph[r].data() : nullptr, 1) != GPSB200_OK) break;
                    const int32_t *pin = nullptr;
                    const double *xin = nullptr;
                    if (r > 0) {                                        // the exact state after slice r-1
                        std::unique_lock<std::mutex> lk(hand[r - 1].mu);
                        hand[r - 1].cv.wait(lk, [&] { return hand[r - 1].ready; });
                        if (hand[r - 1].failed) break;
                        pin = hand[r - 1].prn.data();
                        xin = hand[r - 1].phase.data();
                    }
                    if (gpsb200_slice_finish(ctx, pin, xin, prn_out.data(), ph_out.data(), nullptr) != GPSB200_OK) break;
                    ok = true;
                } while (false);
                {
                    std::lock_guard<std::mutex> lk(hand[r].mu);        // hand on (or release the successor on failure)
                    hand[r].prn = prn_out;
                    hand[r].phase = ph_out;
                    hand[r].failed = !ok;
                    hand[r].ready = true;
                }
                hand[r].cv.notify_all();
                if (ok && gpsb200_slice_wait(ctx) != GPSB200_OK) ok = false;
                if (!ok && ctx) fprintf(stderr, "gpsb200 (device %d): %s\n", r, gpsb200_last_error(ctx));
                if (ctx) gpsb200_destroy(ctx);
                {
                    std::lock_guard<std::mutex> lk(done_mu);
                    done[r] = ok ? 1 : -1;
                }
                done_cv.notify_all();
            });
        }
        if (!fifo_create(8, GPSB200_BLOCK_ELEMS, sample_size)) return 1;       // sdr_iqfile.c:59, sdr.h:24
        bool failed = false;
        for (int r = 0; r < gpus && !failed; r++) {                 // one sink, stream order
            {
                std::unique_lock<std::mutex> lk(done_mu);
                done_cv.wait(lk, [&] { return done[r] != 0; });
                failed = done[r] < 0;
            }
            if (failed) break;
            for (int b = 0; b < lo[r + 1] - lo[r]; b++) {
                if (!start_writer_if_primed(false)) return 1;
                struct iq_buf *iq = fifo_acquire();
                if (!iq) return 1;
                memcpy(sample_size == GPSB200_SC16 ? (void *) iq->data16 : (void *) iq->data8,
                       (char *) slice_host[r] + (size_t) b * blk_bytes, blk_bytes);
                iq->validLength = GPSB200_BLOCK_ELEMS;
                fifo_enqueue(iq);
                queued++;
            }
        }
        for (auto &t : workers) t.join();
        if (failed) return 1;
        if (!start_writer_if_primed(true)) return 1;
        gpsb200_iqfile_stop();
        fifo_destroy();
        for (void *p : slice_host) cudaFreeHost(p);
    }
    gpsb200_scenario_destroy(scn);
    const double dt = now_s() - t0;
    fprintf(stderr, "gpsb200-sim: %d blocks (%d channels) on %d GPU(s) -> %s in %.3f s (%.1f Msamples/s incl. file sink)\n", nblk,
            nchan, gpus, out.c_str(), dt, (double) nblk * GPSB200_BLOCK_SAMPLES / dt / 1e6);
    return 0;
}
