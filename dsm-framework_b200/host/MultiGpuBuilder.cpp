// MultiGpuBuilder.cpp -- see MultiGpuBuilder.h.  Only the C ABI of include/dsmfm.h is used.
#include "MultiGpuBuilder.h"
#include "dsmfm.h"

#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <mutex>
#include <sstream>
#include <thread>
#include <vector>

namespace {

// all threads of a build meet here; a thread that failed poisons the barrier so that nobody waits for it
class Barrier
{
public:
    explicit Barrier(unsigned n) : n_(n) {}
    bool wait(bool ok)
    {
        std::unique_lock<std::mutex> lock(mu_);
        if (!ok) failed_ = true;
        const unsigned long gen = gen_;
        if (++count_ == n_)
        {
            count_ = 0;
            ++gen_;
            cv_.notify_all();
        }
        else
            cv_.wait(lock, [&] { return gen_ != gen; });
        return !failed_;
    }

private:
    std::mutex mu_;
    std::condition_variable cv_;
    unsigned n_, count_ = 0;
    unsigned long gen_ = 0;
    bool failed_ = false;
};

[[noreturn]] void die(std::string const &what)
{
    std::cerr << "builder: " << what << std::endl;
    std::exit(1);
}

} // namespace

MultiGpuBuilder::MultiGpuBuilder(unsigned gpus, unsigned samplerate, bool samples)
    : gpus_(gpus ? gpus : 1), samplerate_(samplerate), samples_(samples)
{
    if (gpus_ > DSMFM_MAX_BLOCKS) die("at most 64 GPUs");
}

void MultiGpuBuilder::Build(uchar const *text, ulong length, std::string const &output, Report &report)
{
    const auto t0 = std::chrono::steady_clock::now();
    const int ndev = dsmfm_device_count();
    if (ndev <= 0) die("no CUDA device available (this builder has no CPU fallback)");
    const unsigned world = gpus_;

    // `getline(...).good()`: a last line without '\n' is dropped (builder.cpp:211)
    ulong use = length;
    while (use > 0 && text[use - 1] != '\n') --use;
    // block r = the bytes [cut[r], cut[r+1]): cut at the first header line at or behind r * use / world, so that a
    // record never straddles two blocks
    std::vector<ulong> cut(world + 1, use);
    cut[0] = 0;
    for (unsigned r = 1; r < world; ++r)
    {
        ulong p = std::max<ulong>(cut[r - 1], (ulong)((unsigned __int128)use * r / world));
        while (p < use && !(text[p] == '>' && (p == 0 || text[p - 1] == '\n')))
        {
            const void *q = std::memchr(text + p, '\n', use - p);
            p = q ? (ulong)((uchar const *)q - text) + 1 : use;
        }
        cut[r] = p;
    }

    std::vector<dsmfm_builder *> b(world, nullptr);
    std::vector<dsmfm_block_info> infos(world);
    std::vector<dsmfm_fasta_info> fasta(world);
    std::vector<void *> text_dev(world, nullptr);
    std::vector<std::vector<uint64_t>> top(world, std::vector<uint64_t>(4096, 0));
    std::vector<uint64_t> hist_all((size_t)world * 256, 0);
    std::vector<dsmfm_shard> shard(world);
    std::vector<dsmfm_pieces> pieces(world);
    std::vector<dsmfm_piece_edge> edges_all;
    std::vector<dsmfm_sa_info> sa_infos(world);
    std::vector<dsmfm_piece_edge> sa_edges((size_t)world * DSMFM_SA_VECTORS);
    std::vector<std::string> errors(world);
    dsmfm_text_plan plan;
    std::memset(&plan, 0, sizeof plan);
    Barrier barrier(world);
    std::mutex mu;

    auto run = [&](unsigned r) {
        const int dev = (int)(r % (unsigned)ndev);
        bool ok = true;
        auto fail = [&](char const *where) {
            if (ok) errors[r] = std::string(where) + ": " + dsmfm_last_error(b[r]);
            ok = false;
        };
        dsmfm_options opt;
        std::memset(&opt, 0, sizeof opt);
        opt.device = dev;
        opt.samplerate = samplerate_;
        opt.shard_index = r;
        opt.shard_count = world;
        opt.shard_span = 1;
        opt.flags = samples_ ? DSMFM_FLAG_KEEP_SA : 0u;
        if (dsmfm_create(&opt, &b[r]) != DSMFM_OK) fail("dsmfm_create");
        // 1. the block: records parsed and transformed on this GPU; its statistics
        if (ok && cut[r + 1] > cut[r] && dsmfm_append_fasta(b[r], text + cut[r], cut[r + 1] - cut[r], 1, &fasta[r]) != DSMFM_OK)
            fail("dsmfm_append_fasta");
        if (ok && dsmfm_block_stats(b[r], &infos[r]) != DSMFM_OK) fail("dsmfm_block_stats");
        if (!barrier.wait(ok)) return;
        // 2. the plan (thread 0 computes, everybody reads)
        if (r == 0)
        {
            const int rc = dsmfm_text_plan_make(infos.data(), world, &plan);
            if (rc != DSMFM_OK)
            {
                errors[0] = rc == DSMFM_EEMPTY ? "can not index empty texts" : "dsmfm_text_plan_make failed";
                ok = false;
            }
            else
                edges_all.resize(0);
        }
        if (!barrier.wait(ok)) return;
        if (plan.n == 0)
        {
            // no documents at all: the reference's one-symbol index (TextCollectionBuilder.cpp:111-119), on one GPU
            if (r == 0)
            {
                dsmfm_builder *one = nullptr;
                dsmfm_index idx;
                dsmfm_options o1;
                std::memset(&o1, 0, sizeof o1);
                o1.device = dev;
                o1.samplerate = samplerate_;
                o1.flags = samples_ ? DSMFM_FLAG_KEEP_SA : 0u;
                if (dsmfm_create(&o1, &one) != DSMFM_OK || dsmfm_finish(one, &idx) != DSMFM_OK ||
                    dsmfm_write_fmi(&idx, output.c_str()) != DSMFM_OK ||
                    (samples_ && dsmfm_write_sa(one, output.c_str()) != DSMFM_OK))
                    errors[0] = std::string("empty collection: ") + dsmfm_last_error(one);
                dsmfm_destroy(one);
            }
            return;
        }
        // 3. pack the block into its slot of this GPU's copy of the packed text
        text_dev[r] = dsmfm_device_alloc(dev, plan.text_bytes);
        if (!text_dev[r])
        {
            errors[r] = "out of device memory for the packed text";
            ok = false;
        }
        if (ok && dsmfm_block_pack(b[r], &plan, r, text_dev[r], top[r].data()) != DSMFM_OK) fail("dsmfm_block_pack");
        if (!barrier.wait(ok)) return;
        //    the exchange: this rank's slot goes to every other GPU (peer copies; NVLink when the devices allow it)
        for (unsigned q = 1; q < world && ok; ++q)
        {
            const unsigned peer = (r + q) % world;
            if (dsmfm_slot_send(b[r], &plan, r, text_dev[r], (int)(peer % (unsigned)ndev), text_dev[peer]) != DSMFM_OK)
                fail("dsmfm_slot_send");
        }
        if (!barrier.wait(ok)) return;
        // 4. the rank's key range of the global suffix order
        std::vector<uint64_t> top_sum(4096, 0);
        for (unsigned q = 0; q < world; ++q)
            for (int i = 0; i < 4096; ++i) top_sum[i] += top[q][i];
        if (ok && dsmfm_build_packed(b[r], &plan, text_dev[r], top_sum.data()) != DSMFM_OK) fail("dsmfm_build_packed");
        if (ok && dsmfm_shard_info(b[r], &shard[r]) != DSMFM_OK) fail("dsmfm_shard_info");
        if (ok && dsmfm_slice_hist(b[r], hist_all.data() + (size_t)r * 256) != DSMFM_OK) fail("dsmfm_slice_hist");
        dsmfm_device_free(dev, text_dev[r]);
        text_dev[r] = nullptr;
        if (!barrier.wait(ok)) return;
        // 5. the rank's share of the wavelet tree and its BitRank directories
        if (ok && dsmfm_pieces_build(b[r], hist_all.data(), world, r, &pieces[r]) != DSMFM_OK) fail("dsmfm_pieces_build");
        if (ok)
        {
            std::lock_guard<std::mutex> g(mu);
            if (edges_all.empty()) edges_all.resize((size_t)world * pieces[r].n_internal);
            std::memcpy(edges_all.data() + (size_t)r * pieces[r].n_internal, pieces[r].edge,
                        sizeof(dsmfm_piece_edge) * pieces[r].n_internal);
        }
        if (!barrier.wait(ok)) return;
        // 6. words and directory entries next to the slice boundaries; 7. the file
        if (ok && dsmfm_pieces_merge(b[r], edges_all.data(), world) != DSMFM_OK) fail("dsmfm_pieces_merge");
        if (ok && dsmfm_pieces_write(b[r], output.c_str(), r == 0) != DSMFM_OK) fail("dsmfm_pieces_write");
        if (!samples_)
        {
            barrier.wait(ok);
            return;
        }
        // 8-11. the same for the .sa samples: slice counts, the rank's share of the five vectors, boundaries, file
        if (ok && dsmfm_sa_slice_info(b[r], &sa_infos[r]) != DSMFM_OK) fail("dsmfm_sa_slice_info");
        if (!barrier.wait(ok)) return;
        if (ok && dsmfm_sa_pieces_build(b[r], sa_infos.data(), world, r, sa_edges.data() + (size_t)r * DSMFM_SA_VECTORS) != DSMFM_OK)
            fail("dsmfm_sa_pieces_build");
        if (!barrier.wait(ok)) return;
        if (ok && dsmfm_sa_pieces_merge(b[r], sa_edges.data(), world) != DSMFM_OK) fail("dsmfm_sa_pieces_merge");
        if (ok && dsmfm_sa_pieces_write(b[r], output.c_str(), r == 0) != DSMFM_OK) fail("dsmfm_sa_pieces_write");
        barrier.wait(ok);
    };

    std::vector<std::thread> threads;
    for (unsigned r = 0; r < world; ++r) threads.emplace_back(run, r);
    for (auto &t : threads) t.join();
    for (unsigned r = 0; r < world; ++r)
        if (!errors[r].empty()) die("GPU rank " + std::to_string(r) + ": " + errors[r]);

    report.records = report.documents = report.bases = report.symbols = report.invalidRecords = report.badHeaders = 0;
    std::ostringstream per;
    uint64_t pos = 0;
    for (unsigned r = 0; r < world; ++r)
    {
        report.records += fasta[r].records;
        report.documents += fasta[r].documents;
        report.bases += fasta[r].bases;
        report.invalidRecords += fasta[r].invalid_records;
        report.badHeaders += fasta[r].bad_headers;
        dsmfm_stats s;
        dsmfm_get_stats(b[r], &s);
        if (shard[r].count && shard[r].rank_begin != pos) die("BWT slices do not tile the suffix order (internal error)");
        pos += shard[r].count;
        per << "  rank " << r << " (device " << r % (unsigned)ndev << "): " << infos[r].documents << " documents, slice ["
            << shard[r].rank_begin << ", " << shard[r].rank_begin + shard[r].count << "), sort " << s.ms_sort << " ms, refinement "
            << s.ms_refine << " ms, wavelet tree " << s.ms_wt << " ms, " << pieces[r].bytes << " bytes of sections\n";
    }
    report.symbols = plan.n ? plan.n : 1;
    if (plan.n && pos != plan.n) die("BWT slices do not cover the suffix order (internal error)");
    report.perGpu = per.str();
    for (unsigned r = 0; r < world; ++r) dsmfm_destroy(b[r]);
    report.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}
