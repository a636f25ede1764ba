// Host-side test tool for the Writer's scores stream (pipeline.hpp; no device code, no CUDA): used by tests/test_scores.py.
//   scores_writer FQ [--chunk N] [--bytes B] [--scores FILE]
// Batcher -> Writer with faked results: read i is reported for gene 0, except that every 7th read (i % 7 == 3) is dropped
// and every 5th (i % 5 == 1) goes through the multi list with genes 0 and 1.  stdout = ssv, OUT1 = the FASTQ file.
// With --scores, read i also carries the record {i % 1000 + 1, i % 997, (i * 2654435761) mod 2^32, its number of
// associations}, and the Writer's fourth output goes to FILE.  PREFAULT pre-faults the mapped outputs as the CLI does.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <string>

#include "pipeline.hpp"

using namespace shkhost;

struct MallocAlloc {
    static void *alloc(size_t n) { return malloc(n); }
    static void free(void *p) { ::free(p); }
};

// shk_host_pack's definition (include/shark_b200.h), restated: the library is not linked here (no -q: codes only)
static void pack_plain(const uint8_t *seq, const uint8_t *, int32_t, uint64_t n, uint64_t *codes, uint32_t *valid)
{
    for (uint64_t g = 0; g < (n + 31) / 32; ++g) {
        uint64_t c = 0;
        uint32_t v = 0;
        for (uint64_t i = g * 32; i < n && i < g * 32 + 32; ++i) {
            const uint32_t ch = seq[i], u = (ch | 0x20u) - 0x61u;
            if (u < 32u && ((0x00080045u >> u) & 1u)) {
                v |= 1u << (i - g * 32);
                c |= (uint64_t)((ch >> 1) & 3u) << (2 * (i - g * 32));
            }
        }
        codes[g] = c;
        valid[g] = v;
    }
}

int main(int argc, char **argv)
{
    if (argc < 2) {
        fprintf(stderr, "usage: scores_writer FQ [--chunk N] [--bytes B] [--scores FILE]\n");
        return 2;
    }
    unsigned chunk = 1000000;
    uint64_t max_bytes = 640000000ull;
    const char *scores = nullptr;
    for (int i = 2; i + 1 < argc; ++i) {
        const std::string a = argv[i];
        if (a == "--chunk") chunk = (unsigned)atol(argv[++i]);
        else if (a == "--bytes") max_bytes = strtoull(argv[++i], nullptr, 10);
        else if (a == "--scores") scores = argv[++i];
    }
    Batcher<MallocAlloc> batcher(argv[1], nullptr, 0, pack_plain);
    if (!batcher.files_ok()) return 1;
    batcher.start();
    std::vector<std::string> legend{"gA", "gB"};
    const char *o1 = getenv("OUT1");
    const int fd1 = o1 ? open(o1, O_RDWR | O_CREAT | O_TRUNC, 0666) : -1;
    const int fd_sc = scores ? open(scores, O_RDWR | O_CREAT | O_TRUNC, 0666) : -1;
    Writer<MallocAlloc> writer(STDOUT_FILENO, fd1, -1, legend, false, fd_sc);
    if (getenv("PREFAULT")) {
        struct stat st;
        const uint64_t expect[3] = {0, fd1 >= 0 && stat(argv[1], &st) == 0 ? (uint64_t)st.st_size * 2 + 4096 : 0, 0};
        writer.start_prefault(expect, 3);
    }
    Chunk<MallocAlloc> ch;
    uint64_t global = 0;
    for (;;) {
        const bool more = batcher.fill(ch, chunk, max_bytes);
        if (batcher.error()) {
            fprintf(stderr, "ERROR %s\n", batcher.error());
            return 3;
        }
        ch.gene16_v.assign(ch.n, 0);
        for (uint32_t r = 0; r < ch.n; ++r, ++global) {
            uint32_t n_assoc = 1;
            if (global % 7 == 3) {
                ch.gene16_v[r] = kGeneNone;
                n_assoc = 0;
            } else if (global % 5 == 1) {
                ch.gene16_v[r] = kGeneMulti;
                ch.multi_v.push_back(AssocPair{r, 0});
                ch.multi_v.push_back(AssocPair{r, 1});
                n_assoc = 2;
            }
            if (scores) {
                const uint32_t rec[4] = {(uint32_t)(global % 1000 + 1), (uint32_t)(global % 997), (uint32_t)(global * 2654435761ull), n_assoc};
                ch.scores_v.insert(ch.scores_v.end(), rec, rec + 4);
            }
        }
        ch.results_from_vectors();
        writer.write(ch);
        if (!more) break;
    }
    writer.flush();
    if (fd1 >= 0) close(fd1);
    if (fd_sc >= 0) close(fd_sc);
    return 0;
}
