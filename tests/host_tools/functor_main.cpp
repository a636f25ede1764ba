// The reference's driver (main.cpp:83-240) restated on top of include/shark_b200_functors.hpp, with -t 1 ordering:
// pass 1 (FastaSplitter batches of 100 records -> KmerBuilder -> BloomfilterFiller), switch_mode(1), pass 2 (canonical
// k-mers of every record -> add_to_kmer, including the `continue` that skips ++nidx), switch_mode(2), then the sample
// stage (FastqSplitter batches of 50 000 reads -> ReadAnalyzer -> ReadOutput).  Parsing is tests/host_tools/fastx.hpp,
// masking, joining and output formatting follow oracle/shark_text.py.  The tests run it where the reference's own
// main.cpp built on the same header (oracle/_ref/shark_hybrid) is not available.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <utility>
#include <vector>

#include "fastx.hpp"
#include "shark_b200_functors.hpp"

static string cstr(const string &s) { return s.substr(0, s.find('\0')); }  // records are C strings (FastqSplitter.hpp:56)

static int base_code(char ch) {
  switch (ch) {
  case 'A': case 'a': return 0;
  case 'C': case 'c': return 1;
  case 'G': case 'g': return 2;
  case 'T': case 't': return 3;
  default: return -1;
  }
}

static uint64_t revcompl(uint64_t kmer, int k) {
  uint64_t rc = 0;
  kmer = ~kmer;
  for (int i = 0; i < k; ++i) {
    rc = (rc << 2) | (kmer & 3);
    kmer >>= 2;
  }
  return rc;
}

// Canonical k-mers of every window of k valid characters, in order; false when there is none (main.cpp:166 `continue`).
static bool canonical_kmers(const string &s, int k, vector<uint64_t> &out) {
  out.clear();
  const uint64_t mask = k == 32 ? ~0ull : ((1ull << (2 * k)) - 1);
  uint64_t kmer = 0;
  int run = 0;
  for (char ch : s) {
    const int c = base_code(ch);
    if (c < 0) {
      run = 0;
      continue;
    }
    kmer = ((kmer << 2) | (uint64_t)c) & mask;
    if (++run >= k) out.push_back(min(kmer, revcompl(kmer, k)));
  }
  return !out.empty();
}

static void usage_fail(const char *msg) {
  fprintf(stderr, "%s\n", msg);
  exit(EXIT_FAILURE);
}

int main(int argc, char **argv) {
  string ref, s1, s2, o1 = "sharked_sample.1", o2 = "sharked_sample.2";
  int k = 17, q = 0;
  double c = 0.6;
  size_t b = 1;
  bool single = false;
  for (int i = 1; i < argc; ++i) {
    const string a = argv[i];
    auto val = [&]() -> string {
      if (i + 1 >= argc) usage_fail("shark : missing argument value");
      return argv[++i];
    };
    if (a == "-r") ref = val();
    else if (a == "-1") s1 = val();
    else if (a == "-2") s2 = val();
    else if (a == "-o") o1 = val();
    else if (a == "-p") o2 = val();
    else if (a == "-k") k = atoi(val().c_str());
    else if (a == "-c") c = atof(val().c_str());
    else if (a == "-b") b = (size_t)atol(val().c_str());
    else if (a == "-q") q = atoi(val().c_str());
    else if (a == "-t") val();  // -t 1 ordering whatever the count
    else if (a == "-s") single = true;
    else usage_fail("shark : unknown argument");
  }
  if (ref.empty() || s1.empty()) usage_fail("shark : missing required files");
  const bool paired = !s2.empty();

  BF bloom(b << 33);  // main.cpp:108
  vector<string> legend_ID;
  {  // pass 1 (main.cpp:128-144)
    KmerBuilder kb(k);
    BloomfilterFiller bff(&bloom);
    shkhost::FastxReader rd(ref.c_str());
    string name, seq, qual;
    bool more = true;
    while (more) {
      auto *texts = new vector<pair<string, string>>();
      while (texts->size() < 100 && (more = rd.read(name, seq, qual) >= 0)) {
        legend_ID.push_back(cstr(name));
        texts->push_back({legend_ID.back(), cstr(seq)});
      }
      if (texts->empty()) {
        delete texts;
        break;
      }
      bff(kb(texts));
    }
  }
  bloom.switch_mode(1);
  {  // pass 2 (main.cpp:154-189)
    shkhost::FastxReader rd(ref.c_str());
    string name, seq, qual;
    vector<uint64_t> kmers;
    int nidx = 0;
    while (rd.read(name, seq, qual) >= 0) {
      const string s = cstr(seq);
      if ((int)s.size() >= k) {
        if (!canonical_kmers(s, k, kmers)) continue;
        bloom.add_to_kmer(kmers, nidx);
      }
      ++nidx;
    }
  }
  bloom.switch_mode(2);

  // sample stage (main.cpp:199-233)
  ReadAnalyzer analyzer(&bloom, legend_ID, k, c, single);
  shkhost::FastxReader r1(s1.c_str());
  std::unique_ptr<shkhost::FastxReader> r2(paired ? new shkhost::FastxReader(s2.c_str()) : nullptr);
  FILE *f1 = fopen(o1.c_str(), "wb");
  FILE *f2 = paired ? fopen(o2.c_str(), "wb") : nullptr;
  if (!f1 || (paired && !f2)) usage_fail("shark : cannot open the output files");
  const signed char mq = (signed char)(q + 33);  // FastqSplitter.hpp:75
  string n1, q1, n2, q2, t1, t2;
  for (;;) {
    vector<elem_t> reads;
    while (reads.size() < 50000) {  // FastqSplitter.hpp:47-93: a failed read ends the batch
      if (r1.read(n1, t1, q1) < 0) break;
      sharseq_t a{cstr(n1), cstr(t1), cstr(q1)}, m;
      if (paired) {
        if (r2->read(n2, t2, q2) < 0) break;
        m = sharseq_t{cstr(n2), cstr(t2), cstr(q2)};
      }
      string text = a.seq, tq = a.qual;
      if (paired) {
        text += 'N' + m.seq;
        tq += '\x1b' + m.qual;
      }
      if (q != 0)  // mask_seq over the quality's length (FastqSplitter.hpp:104-109)
        for (size_t i = 0; i < tq.size() && i < text.size(); ++i)
          if ((signed char)tq[i] < mq) text[i] = (char)(text[i] - 64);
      reads.push_back({text, {a, m}});
    }
    if (reads.empty()) break;
    ReadAnalyzer::output_t out;
    analyzer(reads, out);
    string previd;  // ReadOutput.hpp:37-50, one call per batch
    for (const auto &as : out) {
      const sharseq_t &a = as.second.first, &m = as.second.second;
      fprintf(stdout, "%s %s\n", a.id.c_str(), as.first.c_str());
      if (previd != a.id) {
        fprintf(f1, "@%s\n%s\n+\n%s\n", a.id.c_str(), a.seq.c_str(), a.qual.c_str());
        if (paired) fprintf(f2, "@%s\n%s\n+\n%s\n", m.id.c_str(), m.seq.c_str(), m.qual.c_str());
      }
      previd = a.id;
    }
  }
  fclose(f1);
  if (f2) fclose(f2);
  return 0;
}
