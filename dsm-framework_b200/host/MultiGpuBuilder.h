// MultiGpuBuilder.h -- `builder --gpus N`: ONE index over the reads of one FASTA input, built by N GPUs of one box.
// No counterpart in the reference, whose builder is one process, one thread, one sample (builder.cpp:266,
// README.md:88-91) and which scales the text length by merging 512 MiB batches through backward search
// (incbwt/rlcsa_builder.cpp:245-318).  Here the input is cut at record boundaries into N blocks (block order =
// document order); one host thread per GPU drives the packed-text exchange of include/dsmfm.h -- statistics,
// pack, peer copies of the packed slots over NVLink, key-range sharded sort, the rank's share of the wavelet
// tree -- and writes its share straight into `<output>.fmi`; with samples, its share of `<output>.sa` as well.  The
// threads meet only at host barriers; no GPU ever waits on another GPU's kernel.
#ifndef DSMFM_HOST_MULTIGPUBUILDER_H_
#define DSMFM_HOST_MULTIGPUBUILDER_H_

#include "TextCollection.h"
#include <string>

class MultiGpuBuilder
{
public:
    struct Report
    {
        ulong records, documents, bases, symbols, invalidRecords, badHeaders;
        double seconds; // wall time of Build
        std::string perGpu; // one line per GPU: device, slice, device times
    };
    // gpus: number of ranks; rank r runs on device r modulo the devices present (so that N ranks can be rehearsed
    // on a box with fewer GPUs: the ranks never wait for each other on the device, only at host barriers)
    // samples: also write `<output>.sa`, the suffix-array samples at `samplerate` (the builders keep the suffix array)
    MultiGpuBuilder(unsigned gpus, unsigned samplerate, bool samples = false);
    // text: the whole FASTA input in host memory.  Writes `<output>.fmi` (and `<output>.sa`).  Errors: message on cerr and exit(1),
    // the convention of TextCollectionBuilder.cpp:67-71, 86-91.
    void Build(uchar const *text, ulong length, std::string const &output, Report &report);

private:
    unsigned gpus_, samplerate_;
    bool samples_;
};

#endif
