// hyper_gen.cpp — the host side of the hot path in C++, above the C ABI (include/hypergen_b200.h).
//
// The reference's host is Rust; no Rust toolchain exists in this image, so the drivers that sit
// on top of the FFI are mirrored here with the same names, arguments and file formats:
//
//   utils::get_fasta_files          src/utils.rs:208-221     *.fna, *.fa, *.fasta (each sorted)
//   fastx_reader::read_merge_seq    src/fastx_reader.rs:6-29 sequence lines joined, 'N' per header
//   sketch_cuda::sketch_cuda        src/sketch_cuda.rs:43-117
//   utils::dump_sketch/load_sketch  src/utils.rs:234-258     bincode 1.x Vec<FileSketch>
//   dist::dist                      src/dist.rs:11-63
//   utils::dump_ani_file            src/utils.rs:260-308     stable sort by ANI, reversed, >= threshold
//
// CLI (same flags as src/utils.rs:44-126):
//   hyper-gen sketch -p <dir> -o <out> [-k 21] [-s 1500] [-S 123] [-d 4096] [-C true] [-t 16] [-i false]
//       -i true (--individual): one sketch per FASTA record instead of one per file (hg_group_sketch_fasta_records),
//       named by the record ID (the header text up to the first space or tab), or `<file>#<record index in the file>`
//       for sequence before a file's first header and for an empty ID.
//   hyper-gen dist   -r <ref sketch> -q <query sketch> -o <out> [-a 85.0]
//   hyper-gen search -r <ref sketch> -q <query sketch> -o <out> [-n 10] [-a 0.0]
//       the -n best refs of every query with ANI >= -a (ties by ascending ref index), one line per result,
//       queries in file order.  The refs are split over every visible GPU (hg_group_search_packed); HG_GPUS=n limits it.
//   hyper-gen cluster -r <sketch> -o <out> [-a 95.0]
//       single-linkage clusters at ANI >= -a, one `representative\tmember` line per sketch: clusters by ascending
//       representative (the smallest index of the cluster), members ascending, the representative's own line first.
//       The pairs are split over every visible GPU (hg_group_cluster_packed); HG_GPUS=n limits it.
//   hyper-gen derep -r <sketch> -o <out> [-a 95.0] [-O file|size]
//       greedy dereplication at ANI >= -a: representatives taken in priority order (-O file: file order; -O size:
//       descending hv_norm_2, ties by file index), every other sketch with its closest representative; the lines of
//       `cluster`, each cluster's representative line first.  On one GPU (hg_derep_packed).
//   hyper-gen triangle -r <sketch> -o <out>
//       the ANI of every pair in the PHYLIP lower-triangular layout mash and skani print: n on the first line, then
//       per sketch its name and, tab-separated, its ANI with every earlier sketch (`dist`'s %u.%03u).  The rows are
//       split over every visible GPU (hg_group_ani_matrix_packed); HG_GPUS=n limits it.
// The GPU path is the only path (`-D gpu` is implied): there is no CPU fallback.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <glob.h>
#include <string>
#include <functional>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/hypergen_b200.h"

namespace types {

struct SketchParams {  // src/types.rs:83-113
  std::string path, out_file;
  bool canonical = true;
  uint8_t ksize = 21;
  uint64_t seed = 123, scaled = 1500;
  size_t hv_d = 4096;
  int threads = 16;
  bool individual = false;  // -i: one sketch per record
};

struct FileSketch {  // src/types.rs:224-235
  uint8_t ksize = 21;
  uint64_t scaled = 1500;
  bool canonical = true;
  uint64_t seed = 123;
  uint64_t hv_d = 4096;
  uint8_t hv_quant_bits = 16;
  int32_t hv_norm_2 = 0;
  std::string file_str;
  std::vector<int16_t> hv;
};

struct SketchDist {  // src/types.rs:237-245
  std::string path_ref_sketch, path_query_sketch, out_file;
  float ani_threshold = 85.0f;
};

struct SketchSearch {
  std::string path_ref_sketch, path_query_sketch, out_file;
  uint32_t top_k = 10;
  float ani_min = 0.0f;
};

struct SketchCluster {
  std::string path_sketch, out_file;
  float ani_th = 95.0f;
};

struct SketchDerep {
  std::string path_sketch, out_file;
  float ani_th = 95.0f;
  std::string order = "file";
};

}  // namespace types

[[noreturn]] static void die(const std::string &msg) {
  fprintf(stderr, "hyper-gen: %s\n", msg.c_str());
  exit(1);
}
static void check(int rc, const char *what) {
  if (rc != HG_OK) die(std::string(what) + ": " + hg_last_error());
}

// every visible GPU of the box (the reference drives CudaDevice::new(0) only, sketch_cuda.rs:52); HG_GPUS=n limits it
static hg_group *open_group() {
  int n = 0;
  if (const char *e = getenv("HG_GPUS")) n = atoi(e);
  hg_group *g = nullptr;
  check(hg_group_create(n, nullptr, &g), "hg_group_create");
  return g;
}

namespace utils {

std::vector<std::string> get_fasta_files(const std::string &path_in) {
  // PathBuf::join (utils.rs:210-212) does not double a trailing separator: "dir/" and "dir" both record "dir/x.fna"
  std::string path = path_in;
  while (path.size() > 1 && path.back() == '/') path.pop_back();
  std::vector<std::string> all;
  for (const char *pat : {"*.fna", "*.fa", "*.fasta"}) {
    glob_t g;
    if (glob((path + "/" + pat).c_str(), GLOB_PERIOD, nullptr, &g) == 0)  // the glob crate lets * match a leading dot (MatchOptions default)
      for (size_t i = 0; i < g.gl_pathc; i++) all.emplace_back(g.gl_pathv[i]);  // glob() sorts
    globfree(&g);
  }
  return all;
}

template <class T> static void put(std::string &b, T v) { b.append(reinterpret_cast<const char *>(&v), sizeof(T)); }

void dump_sketch(const std::vector<types::FileSketch> &fs, const std::string &out) {
  std::string b;
  put<uint64_t>(b, fs.size());
  for (const auto &s : fs) {
    put<uint8_t>(b, s.ksize);
    put<uint64_t>(b, s.scaled);
    put<uint8_t>(b, s.canonical ? 1 : 0);
    put<uint64_t>(b, s.seed);
    put<uint64_t>(b, s.hv_d);
    put<uint8_t>(b, s.hv_quant_bits);
    put<int32_t>(b, s.hv_norm_2);
    put<uint64_t>(b, s.file_str.size());
    b += s.file_str;
    put<uint64_t>(b, s.hv.size());
    b.append(reinterpret_cast<const char *>(s.hv.data()), s.hv.size() * 2);
  }
  std::ofstream f(out, std::ios::binary);
  if (!f) die("Dump sketch file failed!");
  f.write(b.data(), (std::streamsize)b.size());
  fprintf(stdout, "Dump sketch file to %s with size %.2f MB\n", out.c_str(), b.size() / 1024.0 / 1024.0);
}

std::vector<types::FileSketch> load_sketch(const std::string &path) {
  std::ifstream f(path, std::ios::binary);
  if (!f) die("Opening sketch file failed!");
  std::string d((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  size_t pos = 0;
  auto get = [&](void *out, size_t n) {
    if (pos + n > d.size()) die("sketch file truncated: " + path);
    memcpy(out, d.data() + pos, n);
    pos += n;
  };
  uint64_t n;
  get(&n, 8);
  std::vector<types::FileSketch> out(n);
  for (auto &s : out) {
    uint8_t c;
    uint64_t len;
    get(&s.ksize, 1); get(&s.scaled, 8); get(&c, 1); s.canonical = c != 0;
    get(&s.seed, 8); get(&s.hv_d, 8); get(&s.hv_quant_bits, 1); get(&s.hv_norm_2, 4);
    get(&len, 8); s.file_str.resize(len); get(&s.file_str[0], len);
    get(&len, 8); s.hv.resize(len); get(s.hv.data(), len * 2);
  }
  return out;
}

}  // namespace utils

namespace fastx_reader {

uint64_t file_size(const std::string &file_name) {
  std::ifstream f(file_name, std::ios::binary | std::ios::ate);
  if (!f) die("Opening .fna files failed: " + file_name);
  return (uint64_t)f.tellg();
}

// the file's bytes as they are, straight into (pinned) staging memory: the GPU does read_merge_seq's job
void read_raw_into(const std::string &file_name, uint8_t *dst, uint64_t size) {
  std::ifstream f(file_name, std::ios::binary);
  if (!f) die("Opening .fna files failed: " + file_name);
  f.read(reinterpret_cast<char *>(dst), (std::streamsize)size);
  if ((uint64_t)f.gcount() != size) die("Reading .fna file failed: " + file_name);
}

std::vector<uint8_t> read_merge_seq(const std::string &file_name) {
  std::ifstream f(file_name, std::ios::binary);
  if (!f) die("Opening .fna files failed: " + file_name);
  std::string d((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  std::vector<uint8_t> out;
  out.reserve(d.size());
  size_t i = 0;
  while (i < d.size()) {
    size_t e = d.find('\n', i);
    size_t end = e == std::string::npos ? d.size() : e;  // line without its '\n'
    if (d[i] == '>') {
      out.push_back('N');
    } else {
      size_t le = end;
      if (le > i && d[le - 1] == '\r') le--;
      out.insert(out.end(), d.begin() + (long)i, d.begin() + (long)le);
    }
    i = e == std::string::npos ? d.size() : e + 1;
  }
  return out;
}

}  // namespace fastx_reader

namespace sketch_cuda {

static double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

void sketch_cuda(const types::SketchParams &params) {
  const auto files = utils::get_fasta_files(params.path);
  const size_t n_file = files.size();
  fprintf(stdout, "Start GPU sketching...\n");
  const bool timing = getenv("HG_CLI_TIMING") != nullptr;  // per-phase wall clock on stderr
  double t_mark = now_s(), t_init = 0, t_stat = 0, t_alloc = 0, t_read = 0, t_gpu = 0, t_collect = 0, t_dump = 0;
  auto lap = [&](double &acc) { const double t = now_s(); acc += t - t_mark; t_mark = t; };
  hg_group *group = open_group();
  hg_ctx *ctx = hg_group_ctx(group, 0);
  const int n_gpus = hg_group_size(group);
  lap(t_init);
  hg_sketch_params p{};
  p.scaled = params.scaled; p.seed = params.seed; p.hv_d = (uint32_t)params.hv_d;
  p.ksize = params.ksize; p.canonical = params.canonical ? 1 : 0;
  const size_t D = params.hv_d;
  std::vector<types::FileSketch> all(params.individual ? 0 : n_file);  // -i: appended record by record
  // By default the raw file bytes go to the GPU, which does read_merge_seq's job itself (hg_sketch_fasta_batch);
  // HG_HOST_PARSE=1 keeps the reference's host-side reader in the loop instead.
  const bool host_parse = getenv("HG_HOST_PARSE") != nullptr;
  if (host_parse && params.individual) die("-i true needs the raw file bytes on the GPU: the host reader (HG_HOST_PARSE=1) has no record mode");
  const int nt_all = std::max(1, params.threads);
  auto parallel = [&](size_t count, const std::function<void(size_t)> &fn) {  // the reference's rayon par_iter over files
    const int nt = (int)std::min<size_t>((size_t)nt_all, std::max<size_t>(count, 1));
    std::vector<std::thread> th;
    for (int t = 0; t < nt; t++)
      th.emplace_back([&, t] { for (size_t i = (size_t)t; i < count; i += (size_t)nt) fn(i); });
    for (auto &x : th) x.join();
  };
  // batches of about 256 MB of file bytes: two page-locked staging buffers of that size (pinning memory costs
  // ~0.4 s per GB, H2D from it runs at the PCIe rate) - the reader threads fill one while the GPU works on the other
  std::vector<uint64_t> fsize(n_file, 0);
  std::vector<std::vector<uint8_t>> parsed(host_parse ? n_file : 0);
  if (host_parse) {
    parallel(n_file, [&](size_t i) { parsed[i] = fastx_reader::read_merge_seq(files[i]); fsize[i] = parsed[i].size(); });
  } else {
    parallel(n_file, [&](size_t i) { fsize[i] = fastx_reader::file_size(files[i]); });
  }
  lap(t_stat);
  const uint64_t batch_bytes = (256ull << 20) * (uint64_t)(host_parse ? 1 : n_gpus);  // per call; the library splits it over the GPUs
  std::vector<std::pair<size_t, size_t>> batches;  // [first, last)
  uint64_t max_batch = 0;
  for (size_t b0 = 0; b0 < n_file;) {
    size_t b1 = b0;
    uint64_t sum = 0;
    do { sum += fsize[b1]; ++b1; } while (b1 < n_file && sum + fsize[b1] <= batch_bytes && b1 - b0 < 65535);
    batches.push_back({b0, b1});
    max_batch = std::max(max_batch, sum);
    b0 = b1;
  }
  uint8_t *stage[2] = {nullptr, nullptr};
  for (int i = 0; i < (batches.size() > 1 ? 2 : 1); i++) check(hg_host_alloc(max_batch + 4096, (void **)&stage[i]), "hg_host_alloc");
  lap(t_alloc);
  std::vector<std::vector<uint64_t>> seg_offs(batches.size());
  std::vector<uint64_t> n_gt(params.individual ? n_file : 0);  // '>' bytes per file: a file holds at most that + 1 records
  auto count_gt = [](const uint8_t *p, uint64_t n) {
    uint64_t c = 0;
    for (const uint8_t *e = p + n; (p = (const uint8_t *)memchr(p, '>', (size_t)(e - p))) != nullptr; ++p) ++c;
    return c;
  };
  auto fill = [&](size_t bi) {  // batch bi into staging buffer bi % 2
    const size_t b0 = batches[bi].first, m = batches[bi].second - b0;
    std::vector<uint64_t> &seg_off = seg_offs[bi];
    seg_off.assign(m + 1, 0);
    for (size_t i = 0; i < m; i++) seg_off[i + 1] = seg_off[i] + fsize[b0 + i];
    uint8_t *dst = stage[bi & 1];
    if (host_parse)
      parallel(m, [&](size_t i) { if (fsize[b0 + i]) memcpy(dst + seg_off[i], parsed[b0 + i].data(), fsize[b0 + i]); });
    else
      parallel(m, [&](size_t i) {
        fastx_reader::read_raw_into(files[b0 + i], dst + seg_off[i], fsize[b0 + i]);
        if (params.individual) n_gt[b0 + i] = count_gt(dst + seg_off[i], fsize[b0 + i]);
      });
  };
  if (!batches.empty()) fill(0);
  lap(t_read);
  for (size_t bi = 0; bi < batches.size(); bi++) {
    const size_t b0 = batches[bi].first, m = batches[bi].second - b0;
    std::thread next;
    if (bi + 1 < batches.size()) next = std::thread(fill, bi + 1);  // overlaps the GPU call below
    const std::vector<uint64_t> &seg_off = seg_offs[bi];
    if (params.individual) {
      uint64_t cap = m;
      for (size_t i = 0; i < m; i++) cap += n_gt[b0 + i];
      if (cap > 0xFFFFFFFFull) cap = 0xFFFFFFFFull;  // the library refuses more records than that anyway
      std::vector<hg_fasta_record> rec(cap);
      std::vector<uint8_t> packed(cap * 2 * D), bits(cap);
      std::vector<int32_t> norm2(cap);
      uint32_t n_rec = 0;
      check(hg_group_sketch_fasta_records(group, stage[bi & 1], seg_off.data(), (uint32_t)m, &p, (uint32_t)cap, rec.data(), packed.data(),
                                          bits.data(), norm2.data(), nullptr, &n_rec),
            "hg_group_sketch_fasta_records");
      for (uint32_t r = 0, index = 0; r < n_rec; r++) {
        index = r && rec[r].file == rec[r - 1].file ? index + 1 : 0;
        types::FileSketch s;
        s.ksize = params.ksize; s.scaled = params.scaled; s.seed = params.seed; s.canonical = params.canonical;
        s.hv_d = D; s.hv_quant_bits = bits[r]; s.hv_norm_2 = norm2[r];
        const char *h = (const char *)stage[bi & 1] + rec[r].name_off;
        s.file_str = rec[r].has_header ? std::string(h, std::find_if(h, h + rec[r].name_len, [](char ch) { return ch == ' ' || ch == '\t'; }))
                                       : std::string();
        if (s.file_str.empty()) s.file_str = files[b0 + rec[r].file] + "#" + std::to_string(index);
        const size_t nbytes = (size_t)bits[r] * D / 8;
        s.hv.resize(nbytes / 2);
        memcpy(s.hv.data(), packed.data() + (size_t)r * 2 * D, nbytes);
        all.push_back(std::move(s));
      }
      if (next.joinable()) next.join();
      continue;
    }
    std::vector<uint8_t> packed(m * 2 * D), bits(m);
    std::vector<int32_t> norm2(m);
    std::vector<uint32_t> nh(m);
    if (host_parse)
      check(hg_sketch_batch(ctx, stage[bi & 1], seg_off.data(), (uint32_t)m, &p, nullptr, packed.data(), bits.data(),
                            norm2.data(), nh.data()), "hg_sketch_batch");
    else
      check(hg_group_sketch_fasta_batch(group, stage[bi & 1], seg_off.data(), (uint32_t)m, &p, nullptr, packed.data(), bits.data(),
                                        norm2.data(), nh.data()), "hg_group_sketch_fasta_batch");
    for (size_t i = 0; i < m; i++) {
      types::FileSketch &s = all[b0 + i];
      s.ksize = params.ksize; s.scaled = params.scaled; s.seed = params.seed; s.canonical = params.canonical;
      s.hv_d = D; s.hv_quant_bits = bits[i]; s.hv_norm_2 = norm2[i]; s.file_str = files[b0 + i];
      const size_t nbytes = (size_t)bits[i] * D / 8;  // hd.rs:146
      s.hv.resize(nbytes / 2);
      memcpy(s.hv.data(), packed.data() + i * 2 * D, nbytes);  // hd.rs:155-157: bytes viewed as i16
    }
    if (next.joinable()) next.join();
  }
  lap(t_gpu);
  check(hg_host_free(stage[0]), "hg_host_free");
  check(hg_host_free(stage[1]), "hg_host_free");
  hg_group_destroy(group);
  lap(t_collect);
  utils::dump_sketch(all, params.out_file);
  lap(t_dump);
  if (timing)
    fprintf(stderr, "[hyper-gen sketch] init %.3f s, stat %.3f, pinned alloc %.3f, first batch read %.3f, GPU calls (+ overlapped reads) %.3f, free %.3f, dump %.3f\n",
            t_init, t_stat, t_alloc, t_read, t_gpu, t_collect, t_dump);
}

}  // namespace sketch_cuda

namespace dist {

struct Stacked { std::vector<uint8_t> packed, bits; std::vector<int32_t> norm; };
static Stacked stack(const std::vector<types::FileSketch> &fs, size_t D) {
  Stacked s;
  s.packed.assign(fs.size() * 2 * D, 0); s.bits.resize(fs.size()); s.norm.resize(fs.size());
  for (size_t i = 0; i < fs.size(); i++) {
    memcpy(s.packed.data() + i * 2 * D, fs[i].hv.data(), std::min(fs[i].hv.size() * 2, 2 * D));
    s.bits[i] = fs[i].hv_quant_bits; s.norm[i] = fs[i].hv_norm_2;
  }
  return s;
}

void dist(const types::SketchDist &sd) {
  const bool if_sym = sd.path_ref_sketch == sd.path_query_sketch;  // dist.rs:13
  auto ref = utils::load_sketch(sd.path_ref_sketch);
  auto qry = if_sym ? ref : utils::load_sketch(sd.path_query_sketch);
  if (ref.empty() || qry.empty()) die("empty sketch file");
  if (ref[0].ksize != qry[0].ksize) die("Ref and query sketches use different kmer sizes!");
  if (ref[0].hv_d != qry[0].hv_d) die("Ref and query sketches use different HV dimensions!");
  const size_t D = ref[0].hv_d, R = ref.size(), Q = qry.size();
  hg_group *group = open_group();
  // The packed rows go to the GPUs as they sit in the sketch file, one block of rows per GPU; decompress_file_sketch (hd.rs:171-232),
  // compute_hv_ani (dist.rs:231-294) and the sort of dump_ani_file (utils.rs:262-269) all run there.
  Stacked rs = stack(ref, D), qs;
  if (!if_sym) qs = stack(qry, D);
  const Stacked &q = if_sym ? rs : qs;
  uint64_t cap = 1 << 20, n_hits = 0;
  std::vector<hg_hit> hits;
  std::vector<uint32_t> milli;  // ANI in thousandths, rounded as `{:.3}` rounds it
  for (;;) {
    hits.resize(cap);
    milli.resize(cap);
    const int rc = hg_group_dist_packed(group, rs.packed.data(), 2 * D, rs.bits.data(), rs.norm.data(), (uint32_t)R, q.packed.data(),
                                        2 * D, q.bits.data(), q.norm.data(), (uint32_t)Q, (uint32_t)D, ref[0].ksize,
                                        sd.ani_threshold, if_sym ? 1 : 0, 1, hits.data(), milli.data(), cap, &n_hits);
    if (rc == HG_E_CAPACITY && n_hits > cap) { cap = n_hits; continue; }
    check(rc, "hg_group_dist_packed");
    break;
  }
  hits.resize(n_hits);
  hg_group_destroy(group);
  std::string csv;
  char buf[64];
  for (size_t t = 0; t < hits.size(); t++) {
    const hg_hit &h = hits[t];
    csv += ref[h.i].file_str; csv += '\t'; csv += qry[h.j].file_str;
    snprintf(buf, sizeof(buf), "\t%u.%03u\n", milli[t] / 1000u, milli[t] % 1000u);
    csv += buf;
  }
  std::ofstream f(sd.out_file, std::ios::binary);
  if (!f) die("Dump ANI file failed!");
  f.write(csv.data(), (std::streamsize)csv.size());
  const double total = if_sym ? (double)R * (double)(Q - 1) / 2.0 : (double)R * (double)Q;
  fprintf(stdout, "Output %zu of %.0f ANIs above threshold %.1f to file %s\n", hits.size(), total,
          (double)sd.ani_threshold, sd.out_file.c_str());
}

}  // namespace dist

namespace search {

void search(const types::SketchSearch &ss) {
  auto ref = utils::load_sketch(ss.path_ref_sketch);
  auto qry = utils::load_sketch(ss.path_query_sketch);
  if (ref.empty() || qry.empty()) die("empty sketch file");
  if (ref[0].ksize != qry[0].ksize) die("Ref and query sketches use different kmer sizes!");
  if (ref[0].hv_d != qry[0].hv_d) die("Ref and query sketches use different HV dimensions!");
  const size_t D = ref[0].hv_d, R = ref.size(), Q = qry.size(), K = ss.top_k;
  const dist::Stacked rs = dist::stack(ref, D), qs = dist::stack(qry, D);
  hg_group *group = open_group();
  std::vector<hg_hit> hits(Q * K);
  std::vector<uint32_t> n_found(Q), milli(Q * K);
  check(hg_group_search_packed(group, rs.packed.data(), 2 * D, rs.bits.data(), rs.norm.data(), (uint32_t)R, qs.packed.data(), 2 * D,
                               qs.bits.data(), qs.norm.data(), (uint32_t)Q, (uint32_t)D, ref[0].ksize, ss.top_k, ss.ani_min, 0,
                               hits.data(), n_found.data(), milli.data()),
        "hg_group_search_packed");
  hg_group_destroy(group);
  std::string out;
  char buf[64];
  size_t lines = 0;
  for (size_t j = 0; j < Q; j++)
    for (size_t r = 0; r < n_found[j]; r++, lines++) {
      const size_t t = j * K + r;
      out += ref[hits[t].i].file_str; out += '\t'; out += qry[j].file_str;
      snprintf(buf, sizeof(buf), "\t%u.%03u\n", milli[t] / 1000u, milli[t] % 1000u);
      out += buf;
    }
  std::ofstream f(ss.out_file, std::ios::binary);
  if (!f) die("Dump search file failed!");
  f.write(out.data(), (std::streamsize)out.size());
  fprintf(stdout, "Output %zu results (top %u per query, ANI >= %.1f) for %zu queries to file %s\n", lines, ss.top_k,
          (double)ss.ani_min, Q, ss.out_file.c_str());
}

}  // namespace search

namespace cluster {

// One `representative\tmember` line per sketch: clusters by ascending representative, the representative's own line
// first, then the members ascending - the key (rep, t != rep, t).
void write_lines(const std::vector<types::FileSketch> &sk, const std::vector<uint32_t> &rep, const std::string &out_file) {
  std::vector<uint32_t> order(rep.size());
  for (size_t t = 0; t < rep.size(); t++) order[t] = (uint32_t)t;
  std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
    return std::make_tuple(rep[a], a != rep[a], a) < std::make_tuple(rep[b], b != rep[b], b);
  });
  std::string out;
  for (uint32_t t : order) {
    out += sk[rep[t]].file_str; out += '\t'; out += sk[t].file_str; out += '\n';
  }
  std::ofstream f(out_file, std::ios::binary);
  if (!f) die("Dump cluster file failed!");
  f.write(out.data(), (std::streamsize)out.size());
}

void cluster(const types::SketchCluster &sc) {
  auto sk = utils::load_sketch(sc.path_sketch);
  if (sk.empty()) die("empty sketch file");
  const size_t D = sk[0].hv_d, n = sk.size();
  const dist::Stacked s = dist::stack(sk, D);
  hg_group *group = open_group();
  std::vector<uint32_t> rep(n);
  uint32_t n_clusters = 0;
  check(hg_group_cluster_packed(group, s.packed.data(), 2 * D, s.bits.data(), s.norm.data(), (uint32_t)n, (uint32_t)D, sk[0].ksize,
                                sc.ani_th, 0, rep.data(), &n_clusters),
        "hg_group_cluster_packed");
  hg_group_destroy(group);
  write_lines(sk, rep, sc.out_file);
  fprintf(stdout, "Output %zu sketches in %u clusters (ANI >= %.1f) to file %s\n", n, n_clusters, (double)sc.ani_th,
          sc.out_file.c_str());
}

}  // namespace cluster

namespace triangle {

// Rows [r0, r1) of the text: sketch i's name, then a tab and ANI(i, j) for every j < i, as `dist` prints it
// (thousandths rounded to nearest even, as ani_milli_kernel rounds them).
static void format_rows(const std::vector<types::FileSketch> &sk, const float *tri, size_t r0, size_t r1, std::string &out) {
  char buf[32];
  for (size_t i = r0; i < r1; i++) {
    out += sk[i].file_str;
    const float *row = tri + i * (i - 1) / 2;
    for (size_t j = 0; j < i; j++) {
      const uint32_t m = (uint32_t)llrint((double)row[j] * 1000.0);
      const int len = snprintf(buf, sizeof(buf), "\t%u.%03u", m / 1000u, m % 1000u);
      out.append(buf, (size_t)len);
    }
    out += '\n';
  }
}

void triangle(const std::string &path_sketch, const std::string &out_file) {
  using clk = std::chrono::steady_clock;
  auto ms = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
  const auto t0 = clk::now();
  auto sk = utils::load_sketch(path_sketch);
  if (sk.empty()) die("empty sketch file");
  const size_t D = sk[0].hv_d, n = sk.size();
  const dist::Stacked s = dist::stack(sk, D);
  const uint64_t entries = (uint64_t)n * (n - 1) / 2;
  float *tri = nullptr;  // page-locked: the bands are copied straight into it
  if (entries) check(hg_host_alloc(entries * 4, (void **)&tri), "hg_host_alloc");
  const auto t1 = clk::now();
  hg_group *group = open_group();
  check(hg_group_ani_matrix_packed(group, s.packed.data(), 2 * D, s.bits.data(), s.norm.data(), (uint32_t)n, s.packed.data(), 2 * D,
                                   s.bits.data(), s.norm.data(), (uint32_t)n, (uint32_t)D, sk[0].ksize, 0, 1, tri, 0),
        "hg_group_ani_matrix_packed");
  hg_group_destroy(group);
  const auto t2 = clk::now();
  // formatting: row ranges of about equal text per thread (row i has i entries)
  const size_t n_th = std::max<size_t>(1, std::min<size_t>(std::thread::hardware_concurrency(), n / 64 + 1));
  std::vector<size_t> cut(n_th + 1, n);
  cut[0] = 0;
  for (size_t k = 1; k < n_th; k++) cut[k] = std::max(cut[k - 1], (size_t)llround((double)n * std::sqrt((double)k / (double)n_th)));
  std::vector<std::string> part(n_th);
  part[0] = std::to_string(n) + "\n";
  std::vector<std::thread> th;
  for (size_t k = 0; k < n_th; k++) th.emplace_back([&, k]() { format_rows(sk, tri, cut[k], cut[k + 1], part[k]); });
  for (auto &t : th) t.join();
  const auto t3 = clk::now();
  std::ofstream f(out_file, std::ios::binary);
  if (!f) die("Dump triangle file failed!");
  for (const std::string &p : part) f.write(p.data(), (std::streamsize)p.size());
  f.close();
  if (tri) hg_host_free(tri);
  const auto t4 = clk::now();
  fprintf(stdout, "Output %zu sketches, %llu ANIs to file %s (ms: load %.1f, GPU %.1f, format %.1f on %zu threads, write %.1f)\n", n,
          (unsigned long long)entries, out_file.c_str(), ms(t0, t1), ms(t1, t2), ms(t2, t3), n_th, ms(t3, t4));
}

}  // namespace triangle

namespace derep {

void derep(const types::SketchDerep &sd) {
  auto sk = utils::load_sketch(sd.path_sketch);
  if (sk.empty()) die("empty sketch file");
  const size_t D = sk[0].hv_d, n = sk.size();
  const dist::Stacked s = dist::stack(sk, D);
  std::vector<uint32_t> order;  // empty: file order
  if (sd.order == "size") {  // descending hv_norm_2 (about hv_d times the sampled hashes: larger genomes first)
    order.resize(n);
    for (size_t t = 0; t < n; t++) order[t] = (uint32_t)t;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return s.norm[a] > s.norm[b]; });
  }
  hg_ctx *ctx = nullptr;
  check(hg_init(0, &ctx), "hg_init");
  std::vector<uint32_t> rep(n);
  uint32_t n_reps = 0;
  check(hg_derep_packed(ctx, s.packed.data(), 2 * D, s.bits.data(), s.norm.data(), (uint32_t)n, (uint32_t)D, sk[0].ksize, sd.ani_th, 0,
                        order.empty() ? nullptr : order.data(), rep.data(), &n_reps),
        "hg_derep_packed");
  hg_destroy(ctx);
  cluster::write_lines(sk, rep, sd.out_file);
  fprintf(stdout, "Output %zu sketches in %u clusters (greedy, ANI >= %.1f) to file %s\n", n, n_reps, (double)sd.ani_th,
          sd.out_file.c_str());
}

}  // namespace derep

int main(int argc, char **argv) {
  if (argc < 2) die("usage: hyper-gen <sketch|dist|search|cluster|derep|triangle> ...");
  const std::string mode = argv[1];
  types::SketchParams sp;
  types::SketchDist sd;
  types::SketchSearch ss;
  types::SketchCluster sc;
  types::SketchDerep sr;
  bool ani_given = false;
  for (int i = 2; i + 1 < argc; i += 2) {
    const std::string k = argv[i], v = argv[i + 1];
    if (k == "-p" || k == "--path") sp.path = v;
    else if (k == "-o" || k == "--out") { sp.out_file = v; sd.out_file = v; ss.out_file = v; sc.out_file = v; sr.out_file = v; }
    else if (k == "-r" || k == "--path_r") { sd.path_ref_sketch = v; ss.path_ref_sketch = v; sc.path_sketch = v; sr.path_sketch = v; }
    else if (k == "-O" || k == "--order") {
      if (v != "file" && v != "size") die("-O must be file or size");
      sr.order = v;
    }
    else if (k == "-q" || k == "--path_q") { sd.path_query_sketch = v; ss.path_query_sketch = v; }
    else if (k == "-n" || k == "--top_k") {
      const long n = atol(v.c_str());
      if (n < 1 || n > 1024) die("-n must be in 1..1024");
      ss.top_k = (uint32_t)n;
    }
    else if (k == "-t" || k == "--thread") sp.threads = atoi(v.c_str());
    else if (k == "-C" || k == "--canonical") sp.canonical = (v == "true" || v == "1");
    else if (k == "-i" || k == "--individual") sp.individual = (v == "true" || v == "1");
    else if (k == "-k" || k == "--ksize") sp.ksize = (uint8_t)atoi(v.c_str());
    else if (k == "-S" || k == "--seed") sp.seed = strtoull(v.c_str(), nullptr, 10);
    else if (k == "-s" || k == "--scaled") sp.scaled = strtoull(v.c_str(), nullptr, 10);
    else if (k == "-d" || k == "--hv_d") sp.hv_d = strtoull(v.c_str(), nullptr, 10);
    else if (k == "-a" || k == "--ani_th") { sd.ani_threshold = (float)atof(v.c_str()); ani_given = true; }
    else if (k == "-D" || k == "--device" || k == "-m" || k == "--sketch_method" || k == "-Q" || k == "--quant_scale") {}
    else die("unknown flag " + k);
  }
  if (mode == "sketch") {
    if (sp.path.empty() || sp.out_file.empty()) die("sketch needs -p and -o");
    sketch_cuda::sketch_cuda(sp);
  } else if (mode == "dist") {
    if (sd.path_ref_sketch.empty() || sd.path_query_sketch.empty() || sd.out_file.empty()) die("dist needs -r -q -o");
    dist::dist(sd);
  } else if (mode == "search") {
    if (ss.path_ref_sketch.empty() || ss.path_query_sketch.empty() || ss.out_file.empty()) die("search needs -r -q -o");
    if (ani_given) ss.ani_min = sd.ani_threshold;
    search::search(ss);
  } else if (mode == "cluster") {
    if (sc.path_sketch.empty() || sc.out_file.empty()) die("cluster needs -r -o");
    if (ani_given) sc.ani_th = sd.ani_threshold;
    cluster::cluster(sc);
  } else if (mode == "derep") {
    if (sr.path_sketch.empty() || sr.out_file.empty()) die("derep needs -r -o");
    if (ani_given) sr.ani_th = sd.ani_threshold;
    derep::derep(sr);
  } else if (mode == "triangle") {
    if (sc.path_sketch.empty() || sc.out_file.empty()) die("triangle needs -r -o");
    triangle::triangle(sc.path_sketch, sc.out_file);
  } else {
    die("unknown subcommand " + mode);
  }
  return 0;
}
