// builder -- drop-in replacement of the reference's `builder` command line
// (builder.cpp:287-471): `builder [-s N] [-v] <input or -> [output]` reads a
// FASTA file and writes `<output or input>.fmi`.  The front end reproduces the
// reference's record handling (builder.cpp:203-262) and per-read transform
// (builder.cpp:60-104, 183-201); the index itself is built on the GPU behind
// TextCollectionBuilder.  There is no CPU fallback.
#include "TextCollectionBuilder.h"
#include "MultiGpuBuilder.h"

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <getopt.h>
#include <iostream>
#include <condition_variable>
#include <mutex>
#include <sstream>
#include <stdexcept>
#include <string>
#include <thread>

namespace {

bool g_verbose = false;
bool g_samples = false; // --samples: also write <output>.sa (the reference's dormant FMIndex::saveSamples)
bool g_fast_exit = true;   // leave through _Exit once the files are written (DSMFM_ORDERLY_EXIT=1: normal teardown)
bool g_host_parse = false; // --host-parse: the reference's per-read loop on the host instead of the GPU front end
unsigned g_gpus = 1;        // --gpus N: one index built by N GPUs (MultiGpuBuilder)

struct Clock
{
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    double seconds() const { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }
};

// Symbol classes of the reference's normalize() (builder.cpp:60-104): lower-case
// acgtn are folded to upper case, ACGTN and the colour-space symbols 0123. pass,
// everything else becomes N and is reported once per record.
struct SymbolTable
{
    unsigned char map[256];
    bool valid[256];
    unsigned char comp[256];
    SymbolTable()
    {
        for (int c = 0; c < 256; ++c) { map[c] = 'N'; valid[c] = false; comp[c] = (unsigned char)c; }
        const char *keep = "ACGTN0123.";
        for (const char *k = keep; *k; ++k) { map[(unsigned char)*k] = (unsigned char)*k; valid[(unsigned char)*k] = true; }
        const char *lower = "acgtn";
        for (const char *k = lower; *k; ++k) { map[(unsigned char)*k] = (unsigned char)(*k - 'a' + 'A'); valid[(unsigned char)*k] = true; }
        comp['A'] = 'T'; comp['T'] = 'A'; comp['C'] = 'G'; comp['G'] = 'C'; // builder.cpp:35-55
    }
};
const SymbolTable kSym;

// doc = reverse(read + '-' + revcomp(read)) = complement(read) + '-' + reverse(read)   (builder.cpp:183-201)
void make_document(std::string const &read, std::string const &name, std::string &doc)
{
    const size_t len = read.size();
    std::string offending;
    doc.resize(2 * len + 1);
    for (size_t i = 0; i < len; ++i)
    {
        const unsigned char raw = (unsigned char)read[i];
        if (!kSym.valid[raw] && offending.find((char)raw) == std::string::npos) offending += (char)raw;
        const unsigned char c = kSym.map[raw];
        doc[i] = (char)kSym.comp[c];
        doc[2 * len - i] = (char)c;
    }
    doc[len] = '-';
    if (!offending.empty())
        std::cerr << "Warning: sequence " << name << " contains invalid symbol(s): " << offending << std::endl;
}

void usage(char const *name)
{
    std::cerr << "usage: " << name << " [options] <input> [output]" << std::endl
              << "Check README or `" << name << " --help' for more information." << std::endl;
}

void help(char const *name)
{
    std::cerr << "usage: " << name << " [options] <input> [output]" << std::endl << std::endl
              << "<input> is the input filename. "
              << "If no output filename is given, the index is stored as <input>.fmi" << std::endl << std::endl
              << "Options:" << std::endl
              << " -s <int>, --sample-rate <int> Sampling rate for the index, a smaller number " << std::endl
              << "                               yields a bigger index but can decrease search " << std::endl
              << "                               time (default: " << TEXTCOLLECTION_DEFAULT_SAMPLERATE << ")." << std::endl
              << " -h, --help                    Display command line options." << std::endl
              << " -v, --verbose                 Print progress information." << std::endl
              << "     --samples                 Also write <output>.sa, the suffix array samples of" << std::endl
              << "                               FMIndex::saveSamples (extension; off in the reference)." << std::endl
              << "     --host-parse              Parse and transform the reads on the host, one InsertText" << std::endl
              << "                               per read as the reference does (default: on the GPU)." << std::endl
              << "     --gpus <int>              Build the one index on <int> GPUs of this box (extension);" << std::endl
              << "                               with --samples every GPU writes its share of <output>.sa." << std::endl;
}

int parse_int_at_least(char const *value, int min, char const *parameter, char const *name)
{
    std::istringstream iss(value);
    int i;
    char c;
    const bool ok = (iss >> i) && !iss.get(c);
    if (!ok || i < min)
    {
        std::cerr << "readaligner: argument of " << parameter << " must be "
                  << (ok ? "" : "of type <int>, and ") << "greater than or equal to " << min << std::endl
                  << "Check README or `" << name << " --help' for more information." << std::endl;
        std::exit(1);
    }
    return i;
}

// After the GPU front end reported symbols that normalize() turns into N: print the reference's warning
// (builder.cpp:94-103) for the first such record, found by re-reading the rows around `offset` on the host.
void warn_invalid(unsigned char const *text, size_t length, size_t offset, unsigned long records)
{
    size_t h = offset; // the header line of the record: the last line start at or before `offset` holding '>'
    std::string name = "undef";
    size_t body = 0;
    while (true)
    {
        size_t ls = h;
        while (ls > 0 && text[ls - 1] != '\n') --ls;
        if (text[ls] == '>')
        {
            size_t e = ls;
            while (e < length && text[e] != '\n') ++e;
            std::string row((char const *)text + ls, e - ls);
            row = row.substr(row.find_first_not_of(" \t", 1));
            name = row.substr(0, row.find_first_of(" \t"));
            body = e + 1;
            break;
        }
        if (ls == 0) break;
        h = ls - 1;
    }
    std::string offending;
    for (size_t i = body; i < length; ++i)
    {
        if (text[i] == '>' && (i == 0 || text[i - 1] == '\n')) break;
        if (text[i] == '\n') continue;
        if (!kSym.valid[text[i]] && offending.find((char)text[i]) == std::string::npos) offending += (char)text[i];
    }
    std::cerr << "Warning: sequence " << name << " contains invalid symbol(s): " << offending << std::endl;
    if (records > 1)
        std::cerr << "Warning: " << records - 1 << " more sequence(s) in this part of the input contain invalid symbols"
                  << " (all turned into N)" << std::endl;
}

// The record loop of build() below, run on the GPU: the file goes to the device in large pieces cut at header
// lines, and TextCollectionBuilder::InsertFasta turns every record into its document there.  A reader thread
// fills one buffer while the GPU works on the other -- and while the CUDA context comes up, which alone takes
// longer than reading a gigabyte.
struct Piece
{
    unsigned char *buf = 0;
    size_t cap = 0, have = 0, use = 0; // bytes held / bytes in front of the last header line (all of them at eof)
    bool eof = false;
};

class PieceReader
{
public:
    PieceReader(FILE *in, size_t cap) : in_(in)
    {
        for (int i = 0; i < 2; ++i)
        {
            piece_[i].buf = (unsigned char *)std::malloc(cap);
            piece_[i].cap = cap;
            if (!piece_[i].buf)
            {
                std::cerr << "builder: unable to allocate the input buffer" << std::endl;
                std::exit(1);
            }
        }
        thread_ = std::thread([this] { run(); });
    }
    ~PieceReader()
    {
        thread_.join();
        std::free(piece_[0].buf);
        std::free(piece_[1].buf);
    }
    // the next piece, or 0 after the last one; the previous piece is released by this call
    Piece *next()
    {
        std::unique_lock<std::mutex> lock(mu_);
        if (taken_ >= 0)
        {
            busy_[taken_] = false;
            taken_ = -1;
            cv_.notify_all();
        }
        cv_.wait(lock, [this] { return ready_ >= 0 || done_; });
        if (ready_ < 0) return 0;
        taken_ = ready_;
        ready_ = -1;
        return &piece_[taken_];
    }

private:
    void run()
    {
        int i = 0;
        size_t carry = 0;
        while (true)
        {
            Piece &p = piece_[i];
            p.have = carry;
            while (true)
            {
                const size_t got = std::fread(p.buf + p.have, 1, p.cap - p.have, in_);
                p.have += got;
                p.eof = got == 0 || std::feof(in_);
                p.use = p.have;
                if (p.eof) break;
                // cut in front of the last header line: the record it opens may continue in the next piece
                p.use = 0;
                for (size_t k = p.have; k > 0;)
                {
                    const void *q = memrchr(p.buf, '>', k);
                    if (!q) break;
                    const size_t at = (size_t)((unsigned char const *)q - p.buf);
                    if (at == 0 || p.buf[at - 1] == '\n')
                    {
                        p.use = at;
                        break;
                    }
                    k = at;
                }
                if (p.use > 0) break;
                // one record larger than the buffer: grow it and keep reading
                unsigned char *bigger = (unsigned char *)std::realloc(p.buf, p.cap * 2);
                if (!bigger)
                {
                    std::cerr << "builder: unable to grow the input buffer" << std::endl;
                    std::exit(1);
                }
                p.buf = bigger;
                p.cap *= 2;
            }
            carry = p.have - p.use;
            Piece &other = piece_[i ^ 1];
            {
                std::unique_lock<std::mutex> lock(mu_);
                cv_.wait(lock, [&] { return !busy_[i ^ 1]; }); // the GPU is done with the other buffer
            }
            if (carry)
            {
                if (other.cap < carry + (p.cap >> 1))
                {
                    std::free(other.buf);
                    other.cap = p.cap;
                    other.buf = (unsigned char *)std::malloc(other.cap);
                    if (!other.buf) std::exit(1);
                }
                std::memcpy(other.buf, p.buf + p.use, carry);
            }
            {
                std::unique_lock<std::mutex> lock(mu_);
                cv_.wait(lock, [this] { return ready_ < 0; });
                busy_[i] = true;
                ready_ = i;
                if (p.eof) done_ = true;
                cv_.notify_all();
                if (p.eof) return;
            }
            i ^= 1;
        }
    }

    FILE *in_;
    Piece piece_[2];
    bool busy_[2] = {false, false};
    int ready_ = -1, taken_ = -1;
    bool done_ = false;
    std::mutex mu_;
    std::condition_variable cv_;
    std::thread thread_;
};

void build_gpu_front_end(FILE *in, std::string const &outputfile, unsigned samplerate, Clock const &wall)
{
    size_t cap = (size_t)4 << 30; // virtual: only the pages a piece really fills are ever touched
    if (const char *e = std::getenv("DSMFM_FASTA_CHUNK_MB")) cap = std::max<size_t>(1, (size_t)std::atol(e)) << 20;
    PieceReader reader(in, cap); // starts reading now, while the device context is created
    TextCollectionBuilder *tcb = new TextCollectionBuilder(samplerate, 1);
    unsigned long bases = 0, records = 0;
    while (Piece *p = reader.next())
    {
        TextCollectionBuilder::FastaReport r;
        tcb->InsertFasta(p->buf, p->use, true, r); // a piece holds whole lines (except, at eof, the dropped last one)
        if (r.badHeaders) // row.substr(npos) in the reference's loop (builder.cpp:215)
            throw std::out_of_range("basic_string::substr: header line without a name");
        if (r.invalidRecords) warn_invalid(p->buf, p->use, r.firstInvalidOffset, r.invalidRecords);
        bases += r.bases;
        records += r.records;
        if (g_verbose)
            std::cerr << "Inserting: " << records << " sequences so far (" << bases / (1024 * 1024) << " MB, elapsed "
                      << wall.seconds() << " s, " << wall.seconds() / 3600 << " hours)" << std::endl;
    }

    std::cerr << "Warning: not thread-safe" << std::endl;
    if (g_verbose)
        std::cerr << "Creating new index with " << records << " sequences, total " << bases << " bytes, "
                  << bases / 1024 << " kb (elapsed " << wall.seconds() << " s, " << wall.seconds() / 3600 << " hours)"
                  << std::endl;
    TextCollection *tc = tcb->InitTextCollection(false, false, 0);
    delete tcb;
    if (g_verbose)
        std::cerr << tc->buildReport() << std::endl
                  << "Saving to file " << outputfile << std::endl
                  << "(total wall-clock time " << wall.seconds() << " s, " << wall.seconds() / 3600 << " hours)"
                  << std::endl;
    tc->save(outputfile);
    if (g_samples) tc->saveSamples(outputfile);
    if (g_fast_exit) return; // the process is about to end: tearing the index down would only cost time
    delete tc;
}

// --gpus N: the whole input is read into (page-locked) host memory, cut into N blocks at record boundaries, and
// N host threads -- one per GPU -- build the one index together (MultiGpuBuilder.h).
void build_multi_gpu(FILE *in, std::string const &outputfile, unsigned samplerate, Clock const &wall)
{
    size_t cap = (size_t)64 << 20, have = 0;
    unsigned char *buf = (unsigned char *)std::malloc(cap);
    while (buf)
    {
        const size_t got = std::fread(buf + have, 1, cap - have, in);
        have += got;
        if (got == 0) break;
        if (have == cap)
        {
            cap *= 2;
            buf = (unsigned char *)std::realloc(buf, cap);
        }
    }
    if (!buf)
    {
        std::cerr << "builder: unable to allocate the input buffer" << std::endl;
        std::exit(1);
    }
    if (g_verbose)
        std::cerr << "Read " << have << " bytes of input (elapsed " << wall.seconds() << " s); building on " << g_gpus
                  << " GPUs" << std::endl;
    std::cerr << "Warning: not thread-safe" << std::endl;
    MultiGpuBuilder mg(g_gpus, samplerate ? samplerate : TEXTCOLLECTION_DEFAULT_SAMPLERATE, g_samples);
    MultiGpuBuilder::Report rep;
    mg.Build(buf, have, outputfile, rep);
    if (rep.badHeaders) throw std::out_of_range("basic_string::substr: header line without a name");
    if (rep.invalidRecords)
        std::cerr << "Warning: " << rep.invalidRecords << " sequence(s) contain invalid symbols (all turned into N)" << std::endl;
    if (g_verbose)
        std::cerr << "Created index with " << rep.documents << " sequences, total " << rep.bases << " bytes, " << rep.symbols
                  << " indexed symbols, in " << rep.seconds << " s on " << g_gpus << " GPU ranks:" << std::endl
                  << rep.perGpu << "Saved to file " << outputfile << ".fmi" << std::endl
                  << "(total wall-clock time " << wall.seconds() << " s, " << wall.seconds() / 3600 << " hours)" << std::endl;
    std::free(buf);
}

void build(std::istream &in, std::string const &outputfile, unsigned samplerate, Clock const &wall)
{
    TextCollectionBuilder *tcb = new TextCollectionBuilder(samplerate, 1);
    unsigned long bases = 0;
    unsigned records = 0;
    std::string seq, name = "undef", row, doc;

    auto flush = [&]() {
        bases += seq.size();
        if (!seq.empty())
        {
            make_document(seq, name, doc);
            tcb->InsertText((uchar const *)doc.c_str(), name);
        }
        seq.clear();
    };

    // `getline(...).good()`: a last line without '\n' sets eofbit and is dropped (builder.cpp:211)
    while (std::getline(in, row).good())
    {
        if (!row.empty() && row[0] == '>')
        {
            // name = header without leading blanks, cut at the first blank (builder.cpp:215-216);
            // like the reference, a header consisting only of '>' throws std::out_of_range
            row = row.substr(row.find_first_not_of(" \t", 1));
            row = row.substr(0, row.find_first_of(" \t"));
            ++records;
            if (row.empty())
            {
                std::ostringstream ss;
                ss << records - 2;
                row = ss.str();
            }
            if (g_verbose && records % 1000000 == 0)
                std::cerr << "Inserting: " << row << " (" << (bases + seq.size()) / (1024 * 1024) << " MB, elapsed "
                          << wall.seconds() << " s, " << wall.seconds() / 3600 << " hours)" << std::endl;
            flush();
            name = row;
        }
        else
            seq.append(row);
    }
    flush();

    std::cerr << "Warning: not thread-safe" << std::endl;
    if (g_verbose)
        std::cerr << "Creating new index with " << records << " sequences, total " << bases << " bytes, "
                  << bases / 1024 << " kb (elapsed " << wall.seconds() << " s, " << wall.seconds() / 3600 << " hours)"
                  << std::endl;

    TextCollection *tc = tcb->InitTextCollection(false, false, 0);
    delete tcb;
    tcb = 0;

    if (g_verbose)
        std::cerr << tc->buildReport() << std::endl
                  << "Saving to file " << outputfile << std::endl
                  << "(total wall-clock time " << wall.seconds() << " s, " << wall.seconds() / 3600 << " hours)"
                  << std::endl;
    tc->save(outputfile);
    if (g_samples) tc->saveSamples(outputfile);
    delete tc;
}

} // namespace

int main(int argc, char **argv)
{
    std::cerr << "Warning: Reversing the string by default" << std::endl;
    if (argc == 1)
    {
        usage(argv[0]);
        return 1;
    }
    unsigned samplerate = 0;
    static struct option long_options[] = {{"sample-rate", required_argument, 0, 's'},
                                           {"help", no_argument, 0, 'h'},
                                           {"verbose", no_argument, 0, 'v'},
                                           {"samples", no_argument, 0, 1000},
                                           {"host-parse", no_argument, 0, 1001},
                                           {"gpus", required_argument, 0, 1002},
                                           {0, 0, 0, 0}};
    int option_index = 0, c;
    // same option string as the reference (builder.cpp:353): -c, -R and -F are accepted by getopt
    // and then rejected, exactly as upstream
    while ((c = getopt_long(argc, argv, "cR:s:F:hv", long_options, &option_index)) != -1)
    {
        switch (c)
        {
        case 's': samplerate = (unsigned)parse_int_at_least(optarg, 1, "-s, --sample-rate", argv[0]); break;
        case 'h': help(argv[0]); return 0;
        case 'v': g_verbose = true; break;
        case 1000: // not in the reference CLI: keeps the suffix array on the GPU and writes the .sa samples too
            g_samples = true;
            setenv("DSMFM_KEEP_SA", "1", 1);
            break;
        case 1001: g_host_parse = true; break;
        case 1002: g_gpus = (unsigned)parse_int_at_least(optarg, 1, "--gpus", argv[0]); break;
        case '?': usage(argv[0]); return 1;
        default: usage(argv[0]); std::abort();
        }
    }
    std::cerr << "Warning: sampling is disabled!" << std::endl;
    if (samplerate && samplerate <= 3)
        std::cerr << "Warning: small samplerates (-s, --sample-rate) may yield infeasible index sizes" << std::endl;
    if (argc - optind < 1)
    {
        std::cerr << "readaligner: no input filename given!" << std::endl;
        usage(argv[0]);
        return 1;
    }
    if (argc - optind > 2)
        std::cerr << "Warning: too many filenames given! Ignoring all but first two." << std::endl;

    const std::string inputfile = argv[optind++];
    std::string outputfile = optind != argc ? std::string(argv[optind++]) : inputfile; // ".fmi" is added by save()

    if (std::getenv("DSMFM_HOST_PARSE")) g_host_parse = true;
    if (std::getenv("DSMFM_ORDERLY_EXIT")) g_fast_exit = false;
    std::ifstream file;
    std::istream *in = &std::cin;
    FILE *fin = stdin;
    if (inputfile != "-")
    {
        if (g_host_parse)
        {
            file.open(inputfile.c_str());
            in = &file;
        }
        else
            fin = std::fopen(inputfile.c_str(), "rb");
    }
    if (g_host_parse ? !in->good() : fin == 0)
    {
        std::cerr << "builder: unable to read input file " << inputfile << std::endl;
        return 1;
    }

    std::cerr << std::fixed;
    std::cerr.precision(2);
    Clock wall;
    if (g_verbose) std::cerr << "Building the forward index:" << std::endl;
    if (g_gpus > 1)
    {
        if (g_host_parse)
        {
            std::cerr << "builder: --gpus can not be combined with --host-parse" << std::endl;
            return 1;
        }
        build_multi_gpu(fin, outputfile, samplerate, wall);
    }
    else if (g_host_parse)
        build(*in, outputfile, samplerate, wall);
    else
        build_gpu_front_end(fin, outputfile, samplerate, wall);
    if (g_verbose)
        std::cerr << "Skipping reverse indexing. Save complete. (total wall-clock time " << wall.seconds() << " s, "
                  << wall.seconds() / 3600 << " hours)" << std::endl;
    if (g_fast_exit)
    {
        // Everything is on disk (save() closed its files).  Unwinding the CUDA context -- tens of gigabytes of
        // pooled device memory -- takes longer than the whole build; the OS reclaims it just the same.
        std::cerr.flush();
        std::fflush(0);
        std::_Exit(0);
    }
    return 0;
}
