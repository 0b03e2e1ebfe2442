// stream.cu — the streaming --usearch_global driver (SURVEY.md §8 f1): FASTA in, --blast6out out.
//
// Replaces, around vsg_group_search, the host loop of the reference's command
//   search_thread_run / search_query      (commands/usearch_global.cpp:376-534)   read a query under mutex_input,
//                                                                                  mask it, search it
//   search_output_results                 (commands/usearch_global.cpp:150-300)   under mutex_output
//   results_show_blast6out_one            (core/results.cpp:221-271)
// by a three-stage pipeline over batches: a reader thread parses the file, the calling thread keeps the GPUs busy
// (upload, DUST, ranking, alignment, accept/reject, hit table), a writer thread formats rows in input order.  At the
// device's rate (hundreds of thousands of queries per second) one query at a time under two mutexes is the
// bottleneck; here parsing batch n+1 and formatting batch n-1 overlap the search of batch n.
#include "vsg_internal.h"

#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace vsg;

namespace {

struct StreamBatch {
  int64_t first = 0;                 // index of the batch's first query in the file
  std::vector<char> cat;             // sequences back to back
  std::vector<int64_t> off;
  std::vector<int32_t> len;
  std::vector<std::string> head;
  std::vector<std::vector<vsg_search_result>> rows;   // of every query, at most --maxhits
  std::vector<int32_t> counts;
  bool last = false;
};

// a bounded hand-over between two stages
class Channel {
 public:
  explicit Channel(size_t cap) : cap_(cap) {}
  void put(std::unique_ptr<StreamBatch> b)
  {
    std::unique_lock<std::mutex> lk(m_);
    cv_.wait(lk, [&] { return q_.size() < cap_ || closed_; });
    if (closed_) { return; }
    q_.push_back(std::move(b));
    cv_.notify_all();
  }
  std::unique_ptr<StreamBatch> get()
  {
    std::unique_lock<std::mutex> lk(m_);
    cv_.wait(lk, [&] { return !q_.empty() || closed_; });
    if (q_.empty()) { return nullptr; }
    std::unique_ptr<StreamBatch> b = std::move(q_.front());
    q_.pop_front();
    cv_.notify_all();
    return b;
  }
  void close()
  {
    std::lock_guard<std::mutex> lk(m_);
    closed_ = true;
    cv_.notify_all();
  }
 private:
  std::mutex m_;
  std::condition_variable cv_;
  std::deque<std::unique_ptr<StreamBatch>> q_;
  size_t cap_;
  bool closed_ = false;
};

double seconds_since(std::chrono::steady_clock::time_point t0)
{
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

// FASTA records of a file, one batch at a time (the reference's parser, core/fasta.cpp / fastx.cpp: a header runs
// to the end of its line and is cut at the first blank unless --notrunclabels; sequence lines are joined, white
// space dropped)
class FastaReader {
 public:
  FastaReader(std::FILE * f, bool notrunc) : f_(f), notrunc_(notrunc), buf_(1 << 22) {}
  // false when the file is exhausted and nothing was read
  bool fill(StreamBatch & b, int want, std::string & err)
  {
    b.cat.clear(); b.off.clear(); b.len.clear(); b.head.clear();
    while (static_cast<int>(b.head.size()) < want) {
      if (!have_header_) {
        if (!next_line()) { break; }
        if (line_.empty()) { continue; }
        if (line_[0] != '>') { err = "FASTA: a sequence line before the first header"; return false; }
        pending_ = header_of(line_);
        have_header_ = true;
      }
      // sequence lines up to the next header
      int64_t const o = static_cast<int64_t>(b.cat.size());
      bool more = false;
      while (next_line()) {
        if (!line_.empty() && line_[0] == '>') { more = true; break; }
        for (char ch : line_) { if (ch != ' ' && ch != '\t' && ch != '\r') { b.cat.push_back(ch); } }
      }
      int64_t const l = static_cast<int64_t>(b.cat.size()) - o;
      if (l > 0x7fffffff) { err = "FASTA: a sequence longer than 2^31"; return false; }
      b.off.push_back(o); b.len.push_back(static_cast<int32_t>(l)); b.head.push_back(pending_);
      if (more) { pending_ = header_of(line_); have_header_ = true; } else { have_header_ = false; }
      if (!more) { break; }
    }
    b.cat.push_back('\0');
    return !b.head.empty();
  }
 private:
  std::string header_of(const std::string & line) const
  {
    size_t e = line.size();
    if (!notrunc_) { for (size_t i = 1; i < line.size(); i++) { if (line[i] == ' ' || line[i] == '\t') { e = i; break; } } }
    return line.substr(1, e - 1);
  }
  bool next_line()
  {
    line_.clear();
    for (;;) {
      if (pos_ == end_) {
        end_ = std::fread(buf_.data(), 1, buf_.size(), f_);
        pos_ = 0;
        if (end_ == 0) { return !line_.empty() || got_partial_(); }
      }
      char const * const s = buf_.data() + pos_;
      char const * const nl = static_cast<char const *>(std::memchr(s, '\n', end_ - pos_));
      if (nl == nullptr) { line_.append(s, end_ - pos_); pos_ = end_; partial_ = true; continue; }
      line_.append(s, static_cast<size_t>(nl - s));
      pos_ += static_cast<size_t>(nl - s) + 1;
      partial_ = false;
      if (!line_.empty() && line_.back() == '\r') { line_.pop_back(); }
      return true;
    }
  }
  bool got_partial_() { bool const p = partial_; partial_ = false; return p; }
  std::FILE * f_;
  bool notrunc_;
  std::vector<char> buf_;
  size_t pos_ = 0, end_ = 0;
  bool partial_ = false;
  std::string line_, pending_;
  bool have_header_ = false;
};

}  // namespace

extern "C" int vsg_usearch_stream(vsg_group * g, const char * const * target_labels, const char * query_fasta,
                                  const vsg_search_opts * opts, int qmask_dust, int notrunclabels, int batch_queries,
                                  int64_t maxhits, int output_no_hits, const char * blast6out_path, vsg_stream_stats * stats)
{
  if (g == nullptr || target_labels == nullptr || query_fasta == nullptr || opts == nullptr || blast6out_path == nullptr) {
    Error::set("vsg_usearch_stream: null argument");
    return VSG_EINVAL;
  }
  if (batch_queries < 1) { batch_queries = 65536; }
  if (maxhits <= 0) { maxhits = INT64_MAX; }
  std::FILE * fin = std::fopen(query_fasta, "rb");
  if (fin == nullptr) { Error::set(std::string("vsg_usearch_stream: cannot open ") + query_fasta); return VSG_EINVAL; }
  std::FILE * fout = std::fopen(blast6out_path, "wb");
  if (fout == nullptr) { std::fclose(fin); Error::set(std::string("vsg_usearch_stream: cannot write ") + blast6out_path); return VSG_EINVAL; }

  auto const t_wall = std::chrono::steady_clock::now();
  vsg_stream_stats st{};
  Channel parsed(2), searched(2);
  std::string reader_err;
  std::thread reader([&] {
    FastaReader fr(fin, notrunclabels != 0);
    int64_t first = 0;
    for (;;) {
      auto const t0 = std::chrono::steady_clock::now();
      std::unique_ptr<StreamBatch> b(new StreamBatch());
      bool const ok = fr.fill(*b, batch_queries, reader_err);
      st.parse_s += seconds_since(t0);
      if (!ok) { break; }
      b->first = first;
      first += static_cast<int64_t>(b->head.size());
      parsed.put(std::move(b));
    }
    std::unique_ptr<StreamBatch> e(new StreamBatch());
    e->last = true;
    parsed.put(std::move(e));
  });
  std::thread writer([&] {
    std::string out;
    for (;;) {
      std::unique_ptr<StreamBatch> b = searched.get();
      if (b == nullptr || b->last) { break; }
      auto const t0 = std::chrono::steady_clock::now();
      out.clear();
      char row[256];
      size_t const nq = b->head.size();
      for (size_t q = 0; q < nq; q++) {
        int64_t const n = b->counts[q];
        if (n > 0) { st.matched++; }
        if (n == 0 && output_no_hits != 0) {
          out += b->head[q]; out += "\t*\t0.0\t0\t0\t0\t0\t0\t0\t0\t-1\t0\n";   // results.cpp:248-250
          st.rows++;
        }
        for (int64_t j = 0; j < n; j++) {
          vsg_search_result const & r = b->rows[q][static_cast<size_t>(j)];
          int const qstart = r.strand != 0 ? r.query_length : 1, qend = r.strand != 0 ? 1 : r.query_length;
          out += b->head[q]; out += '\t'; out += target_labels[r.target];
          int const w = std::snprintf(row, sizeof row, "\t%.1f\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\n", r.id, r.internal_alignment_length,
                                      r.mismatches, r.internal_gaps, qstart, qend, 1, r.target_length, -1, 0);
          out.append(row, static_cast<size_t>(w));
          st.rows++;
        }
      }
      std::fwrite(out.data(), 1, out.size(), fout);
      st.write_s += seconds_since(t0);
    }
  });

  int rc = VSG_OK;
  for (;;) {
    std::unique_ptr<StreamBatch> b = parsed.get();
    if (b == nullptr || b->last) { break; }
    auto const t0 = std::chrono::steady_clock::now();
    int64_t const nq = static_cast<int64_t>(b->head.size());
    b->rows.assign(static_cast<size_t>(nq), {});
    b->counts.assign(static_cast<size_t>(nq), 0);
    rc = group_search_rows(g, b->cat.data(), b->off.data(), b->len.data(), nq, qmask_dust, opts, maxhits, b->rows.data(),
                           b->counts.data(), nullptr);
    st.search_s += seconds_since(t0);
    if (rc != VSG_OK) { break; }
    st.queries += nq; st.batches++;
    st.nucleotides += static_cast<int64_t>(b->cat.size()) - 1;
    searched.put(std::move(b));
  }
  if (rc != VSG_OK) { parsed.close(); }   // unblocks the reader
  {
    std::unique_ptr<StreamBatch> e(new StreamBatch());
    e->last = true;
    searched.put(std::move(e));
  }
  reader.join();
  writer.join();
  std::fclose(fin);
  if (std::fclose(fout) != 0 && rc == VSG_OK) { Error::set("vsg_usearch_stream: write error"); rc = VSG_EINVAL; }
  if (rc == VSG_OK && !reader_err.empty()) { Error::set("vsg_usearch_stream: " + reader_err); rc = VSG_EINVAL; }
  st.wall_s = seconds_since(t_wall);
  if (stats != nullptr) { *stats = st; }
  return rc;
}
