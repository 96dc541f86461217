// `pRIblast db` front-end on top of libpriblast_acc.so: same options and defaults as the reference
// (main.cpp:43-73, db_construction_parameters.cpp:32-78), same five output files (SURVEY §2.2).
// The per-sequence OpenMP/MPI loop of DbConstruction::CalculateAccessibility (db_construction.cpp:170-229)
// becomes ONE prib_acc_run call per GPU; the block/heap/dynamic distributors (-a) all map to the
// length-balanced partitioner over the GPUs of this box (db_format.h lpt_partition); output order is the
// FASTA order, i.e. what the reference emits with -np 1 and -a heap|block.
//
// Process model: one WORKER PROCESS per GPU (the reference: one MPI rank per node), forked before the first CUDA
// call and pinned to its device through CUDA_VISIBLE_DEVICES, so the CUDA start-up of eight B200s (0.55 s each,
// 5.4 s when one process opens all of them: profiles/r1/cuda_init_8gpu.txt) runs in parallel.  Every worker writes
// the records of its sequences straight into <db>.acc at their final offsets (pwrite; the record sizes are known
// from the lengths), so there is no gather step at all.  The parent builds <db>.seq/.ind/.nam/.bas meanwhile (suffix
// arrays on the last GPU).
//
// -d may list several minimum accessible lengths (`-d 5,8,12`).  Then one accessibility context per worker computes all
// of them (prib_acc_create_lengths: the inside and outside passes are shared), and the front-end writes one complete
// database per length, <db>_d<delta>, each byte-identical to a run with that -d alone.  The suffix arrays, the hash,
// <db>.seq/.ind and <db>.nam are built once and copied.
#include <fcntl.h>
#include <getopt.h>
#include <signal.h>
#include <sys/mman.h>
#include <sys/wait.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <chrono>
#include <cstring>
#include <future>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/priblast_acc.h"
#include "db_format.h"

using namespace prib;

static int die(const std::string &msg) {
  std::fprintf(stderr, "%s\n", msg.c_str());
  return 1;
}

// -d: one integer (read with atoi, as the reference does), or a comma-separated, strictly increasing list
static bool parse_lengths(const char *arg, std::vector<int> &out, std::string &err) {
  out.clear();
  if (!std::strchr(arg, ',')) {
    out.push_back(std::atoi(arg));
    return true;
  }
  for (const char *p = arg;;) {
    char *end = nullptr;
    const long v = std::strtol(p, &end, 10);
    if (end == p || (*end != ',' && *end != 0) || v < INT32_MIN || v > INT32_MAX) {
      err = std::string("Error: -d must be an integer or a comma-separated list of integers, not '") + arg + "'";
      return false;
    }
    out.push_back((int)v);
    if (*end == 0) break;
    p = end + 1;
  }
  if ((int)out.size() > PRIB_MAX_LENGTHS) {
    err = "Error: -d takes at most " + std::to_string(PRIB_MAX_LENGTHS) + " values";
    return false;
  }
  for (size_t l = 1; l < out.size(); l++)
    if (out[l] <= out[l - 1]) {
      err = "Error: the -d values must be strictly increasing";
      return false;
    }
  return true;
}

static bool copy_file(const std::string &from, const std::string &to, std::string &err) {
  std::FILE *in = std::fopen(from.c_str(), "rb");
  std::FILE *out = in ? std::fopen(to.c_str(), "wb") : nullptr;
  bool ok = in && out;
  std::vector<char> buf(1 << 20);
  while (ok) {
    const size_t n = std::fread(buf.data(), 1, buf.size(), in);
    ok = std::fwrite(buf.data(), 1, n, out) == n;
    if (n < buf.size()) break;
  }
  ok = ok && !std::ferror(in);
  if (in) std::fclose(in);
  if (out && std::fclose(out) != 0) ok = false;
  if (!ok) err = "Error: can't copy " + from + " to " + to;
  return ok;
}

// <db>.ind: the suffix array of every page is built on GPU 0 (prib_suffix_array replaces sais(),
// db_construction.cpp:330-335)
static bool gpu_suffix_array(const uint8_t *text, int n, std::vector<int32_t> &sa, std::string &err) {
  sa.resize((size_t)std::max(n, 0));
  if (prib_suffix_array(text, n, sa.data(), 0) != PRIB_OK) {
    err = std::string("Error: suffix array: ") + prib_last_error();
    return false;
  }
  return true;
}

// PRIB_DB_TIMING=1: wall time of every stage on stderr
struct StageTimer {
  bool on = std::getenv("PRIB_DB_TIMING") != nullptr;
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  void lap(const char *what) {
    const auto now = std::chrono::steady_clock::now();
    if (on) std::fprintf(stderr, "[db] %-28s %9.3f s\n", what, std::chrono::duration<double>(now - t).count());
    t = now;
  }
};

// GPUs of this box without touching CUDA: initialising the CUDA driver costs ~0.55 s + ~0.7 s per additional visible
// B200 (5.4 s with 8 on an NVSwitch box, profiles/r1/cuda_init_8gpu.txt), so the front-end decides how many GPUs a
// job is worth BEFORE the first CUDA call and hides the rest through CUDA_VISIBLE_DEVICES.
static int count_device_nodes() {
  int n = 0;
  for (int k = 0; k < 64; k++) {
    const std::string node = "/dev/nvidia" + std::to_string(k);
    if (FILE *f = std::fopen(node.c_str(), "rb")) {
      std::fclose(f);
      ++n;
    } else if (access(node.c_str(), F_OK) == 0) {
      ++n;
    }
  }
  return n;
}

static void usage() {
  std::printf(
      "pRIblast-b200 db: database construction with GPU accessibility\n"
      "usage: pRIblast_b200 db -i InputFastaFile -o OutputDbName [-r RepeatMaskingStyle] [-s LookupTableSize]\n"
      "                        [-w MaximalSpan] [-d MinAccessibleLength[,...]] [-c ChunkSize] [-a block|heap|dynamic]\n"
      "                        [-p TmpPath] [-m auto|fp64|exact]\n"
      "defaults: -r 0 -s 8 -w 70 -d 5 -a heap -c INT_MAX   (reference: main.cpp:43-73)\n"
      "ranges: -w 1..1000, -d 2..1000 (-d may exceed -w); above -w 200, auto and fp64 run the FP64 wide-span engine\n"
      "   (.acc within 1e-4 kcal/mol of the reference; sequences whose values leave its range are recomputed by the\n"
      "   exact engine)\n"
      "-m (extension; also PRIB_ACC_MODE): auto = FP32 span-scaled engine with FP64 re-run (default; .acc within\n"
      "   1e-4 kcal/mol of the reference), fp64, exact = the reference's own arithmetic on the GPU (.acc, hence\n"
      "   the whole database and the ris output, byte-identical to a reference built WITHOUT FMA contraction,\n"
      "   i.e. -ffp-contract=off or no -march; the upstream Makefile's -march=native build differs from that in\n"
      "   the last bit of 65 %% of the values, max 4.8e-7 kcal/mol; ~50x slower than auto)\n"
      "-d 5,8,12 (extension): up to 32 strictly increasing lengths computed together (the inside and outside passes\n"
      "   are shared); writes one complete database per length, OutputDbName_d5, OutputDbName_d8, ..., each identical\n"
      "   to a run with that -d alone\n"
      "environment: PRIB_NUM_GPUS=n limits the number of GPUs (default: every visible one, one worker process each)\n");
}

int main(int argc, char *argv[]) {
  if (argc == 1 || std::strcmp(argv[1], "-h") == 0) {
    usage();
    return 0;
  }
  if (std::strcmp(argv[1], "db") != 0) {
    std::printf("usage: pRIblast_b200 [-h] db options   (the `ris` step stays the reference binary)\n");
    return 0;
  }
  std::string input, db, tmp_path, alg = "heap";
  std::string mode = std::getenv("PRIB_ACC_MODE") ? std::getenv("PRIB_ACC_MODE") : "auto";
  DbParams prm;
  std::vector<int> lengths(1, prm.min_accessible_length);
  std::string err;
  int c;
  optind = 1;
  while ((c = getopt(argc - 1, argv + 1, "i:o:r:s:w:d:t:p:a:c:m:")) != -1) {
    switch (c) {
      case 'i': input = optarg; break;
      case 'o': db = optarg; break;
      case 'r': prm.repeat_flag = std::atoi(optarg); break;
      case 's': prm.hash_size = std::atoi(optarg); break;
      case 'w': prm.maximal_span = std::atoi(optarg); break;
      case 'd':
        if (!parse_lengths(optarg, lengths, err)) return die(err);
        break;
      case 'p': tmp_path = optarg; break;  // accepted; there are no temp files any more
      case 'a': alg = optarg; break;
      case 'c': prm.chunk_size = std::atoi(optarg); break;
      case 'm': mode = optarg; break;
      default: return die("Error: invalid argument");  // incl. -t, as in the reference
    }
  }
  if (alg != "block" && alg != "heap" && alg != "dynamic") return die("Error: parallel algorithm not supported");
  if (mode != "auto" && mode != "fp64" && mode != "exact") return die("Error: -m must be auto, fp64 or exact");
  const int acc_mode = mode == "exact" ? 2 : mode == "fp64" ? 1 : 0;

  std::vector<std::string> names, seqs;
  StageTimer timer;
  if (!read_fasta(input, names, seqs, err)) return die(err);
  timer.lap("read FASTA");
  if (db.empty()) return die("Error: -o option is required");                                   // raccess.hpp:42-45
  for (int d : lengths)
    if (d <= 1) return die("Error: -d option must be greater than 1");   // raccess.hpp:47-50
  if (prm.repeat_flag < 0 || prm.repeat_flag > 2) return die("Error: -r option must be 0, 1, or 2");
  prm.min_accessible_length = lengths[0];
  const size_t nlen = lengths.size();
  for (size_t k = 0; k < seqs.size(); k++)
    if ((int)seqs[k].size() < lengths.back())
      return die("Error: sequence " + names[k] + " is shorter than the minimum accessible length (-d): the "
                 "reference writes a corrupt record for it (raccess.cpp:449-450); refusing");
  // one database per length: <db> itself for one length, <db>_d<delta> for a list
  std::vector<std::string> dbs;
  for (int d : lengths) dbs.push_back(nlen == 1 ? db : db + "_d" + std::to_string(d));
  auto write_copies = [&](std::string &e) {  // <dbs[0]>.seq/.ind, built once, for the other databases
    for (size_t l = 1; l < nlen; l++)
      for (const char *ext : {".seq", ".ind"})
        if (!copy_file(dbs[0] + ext, dbs[l] + ext, e)) return false;
    return true;
  };
  auto write_nam_bas = [&](std::string &e) {
    for (size_t l = 0; l < nlen; l++) {
      DbParams pl = prm;
      pl.min_accessible_length = lengths[l];
      if (!write_nam(dbs[l], names, e) || !write_bas(dbs[l], pl, e)) return false;
    }
    return true;
  };

  // ---- accessibility on the GPUs ---------------------------------------------------------------
  const bool formats_only = std::getenv("PRIB_DB_FORMATS_ONLY") != nullptr;  // test switch: no .acc, no GPU
  // record k of <db>.acc starts at rec_off[l][k] (raccess.cpp:447-481: 8 + 4 (2L - delta + 1) bytes per sequence)
  std::vector<std::vector<int64_t>> rec_off(nlen, std::vector<int64_t>(seqs.size() + 1, 0));
  for (size_t l = 0; l < nlen; l++)
    for (size_t k = 0; k < seqs.size(); k++)
      rec_off[l][k + 1] = rec_off[l][k] + prib_acc_record_bytes((int32_t)seqs[k].size(), lengths[l]);
  bool ok = true;
  bool workers_ok = true;
  if (!formats_only) {
    // the devices we may use: the caller's CUDA_VISIBLE_DEVICES list if there is one, else the /dev/nvidiaN nodes
    // (counted without touching CUDA: nothing in this process may initialise it before the fork)
    std::vector<std::string> devs;
    if (const char *cv = std::getenv("CUDA_VISIBLE_DEVICES")) {
      std::string item;
      for (const char *q = cv;; ++q) {
        if (*q == ',' || *q == 0) {
          if (!item.empty()) devs.push_back(item);
          item.clear();
          if (*q == 0) break;
        } else {
          item += *q;
        }
      }
    } else {
      const int nodes = count_device_nodes();
      for (int k = 0; k < nodes; k++) devs.push_back(std::to_string(k));
    }
    int fixed_gpus = 0;  // PRIB_NUM_GPUS=n: exactly n workers, all started at once (scaling measurements)
    if (const char *e = std::getenv("PRIB_NUM_GPUS")) fixed_gpus = std::max(1, std::atoi(e));
    if (fixed_gpus > 0 && (size_t)fixed_gpus < devs.size()) devs.resize((size_t)fixed_gpus);
    if (devs.empty()) return die("Error: no CUDA device available (there is no CPU path)");
    for (size_t l = 0; l < nlen; l++) {  // <db>.acc at its final size; the workers fill it in place
      const int fd = open((dbs[l] + ".acc").c_str(), O_CREAT | O_TRUNC | O_WRONLY, 0644);
      if (fd < 0 || ftruncate(fd, (off_t)rec_off[l][seqs.size()]) != 0) return die("Error: can't open " + dbs[l] + ".acc");
      close(fd);
    }
    // Work units: the sequences longest first (the order of SortSequences, utils.cpp:53-60: neighbours in a device
    // batch have similar lengths), cut into chunks of ~4 M nt.  The workers claim chunks from a shared counter — the
    // reference's `-a dynamic` distributor (the MPI RMA counter of db_construction.cpp:85-95, 191-197) in shared memory.
    std::vector<int> order(seqs.size());
    for (size_t k = 0; k < order.size(); k++) order[k] = (int)k;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b2) { return seqs[(size_t)a].size() > seqs[(size_t)b2].size(); });
    std::vector<size_t> chunk_begin(1, 0);
    {
      const int64_t target = 4 << 20;
      int64_t acc_nt = 0;
      for (size_t k = 0; k < order.size(); k++) {
        acc_nt += (int64_t)seqs[(size_t)order[k]].size();
        if (acc_nt >= target && k + 1 < order.size()) {
          chunk_begin.push_back(k + 1);
          acc_nt = 0;
        }
      }
      chunk_begin.push_back(order.size());
    }
    const int nchunks = (int)chunk_begin.size() - 1;
    struct Shared {  // one page of MAP_SHARED memory
      int next_chunk, done_chunks, ready, failed, sa_claimed, sa_done;
      long long nt_done;
      double t_first_ready, t_last_ready;
    };
    Shared *sh = (Shared *)mmap(nullptr, 4096, PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS, -1, 0);
    if (sh == MAP_FAILED) return die("Error: mmap failed");
    std::memset(sh, 0, sizeof(*sh));
    const auto t_start = std::chrono::steady_clock::now();
    auto since_start = [&]() { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count(); };
    std::fflush(nullptr);

    auto worker_main = [&](int d) {  // ---- worker d: its own process, its own CUDA context on its own device
      setenv("CUDA_VISIBLE_DEVICES", devs[(size_t)d].c_str(), 1);
      auto fail_w = [&](const std::string &msg) {
        std::fprintf(stderr, "Error: GPU %s: %s\n", devs[(size_t)d].c_str(), msg.c_str());
        __atomic_store_n(&sh->failed, 1, __ATOMIC_SEQ_CST);
        _exit(1);
      };
      // <db>.seq / <db>.ind need only the sequences: the first worker that gets here builds them in a second thread
      // of its process, suffix arrays on its GPU (one CUDA start-up per device)
      std::string err_si;
      std::future<bool> seq_ind;
      if (__atomic_exchange_n(&sh->sa_claimed, 1, __ATOMIC_SEQ_CST) == 0)
        seq_ind = std::async(std::launch::async, [&]() {
          StageTimer t_si;
          const bool ok_si = write_seq_ind(dbs[0], seqs, prm, err_si, gpu_suffix_array) && write_copies(err_si);
          t_si.lap("  worker: .seq/.ind (SA on GPU, hash) [thread]");
          return ok_si;
        });
      StageTimer wt;
      prib_acc_params ap;
      std::memset(&ap, 0, sizeof(ap));
      ap.maximal_span = prm.maximal_span;
      ap.device = 0;
      ap.mode = acc_mode;
      prib_ctx *ctx = nullptr;
      if (prib_acc_create_lengths(&ctx, &ap, (int32_t)nlen, lengths.data()) != PRIB_OK) fail_w(prib_last_error());
      wt.lap("  worker: context (CUDA init, tables)");
      {
        const double tr = since_start();
        if (__atomic_fetch_add(&sh->ready, 1, __ATOMIC_SEQ_CST) == 0) sh->t_first_ready = tr;
        sh->t_last_ready = tr;
      }
      std::vector<int> fds(nlen);
      for (size_t l = 0; l < nlen; l++) {
        fds[l] = open((dbs[l] + ".acc").c_str(), O_WRONLY);
        if (fds[l] < 0) fail_w("can't open " + dbs[l] + ".acc");
      }
      // two page-locked result images: while the records of chunk c go to the file (a second thread: memcpy + pwrite),
      // the GPU already works on chunk c + 1
      struct Slot {
        float *image = nullptr;
        int64_t floats = 0;
        std::vector<int32_t> sl;
        std::vector<int64_t> ao, co;
        std::future<bool> writing;
      } slot[2];
      std::vector<const char *> sp;
      int mine = 0;
      for (int cur = 0;; cur ^= 1) {
        const int ch = __atomic_fetch_add(&sh->next_chunk, 1, __ATOMIC_SEQ_CST);
        if (ch >= nchunks) break;
        Slot &S = slot[cur];
        if (S.writing.valid() && !S.writing.get()) fail_w("short write on an .acc file");
        const size_t k0 = chunk_begin[(size_t)ch], k1 = chunk_begin[(size_t)ch + 1], n = k1 - k0;
        sp.resize(n);
        S.sl.resize(n);
        S.ao.resize(nlen * n);
        S.co.resize(nlen * n);
        int64_t total = 0;  // floats of one length's image; the images of the lengths lie back to back
        for (size_t k = 0; k < n; k++) {
          const std::string &sq = seqs[(size_t)order[k0 + k]];
          sp[k] = sq.data();
          S.sl[k] = (int32_t)sq.size();
          S.ao[k] = total;
          S.co[k] = total + S.sl[k];
          total += 2 * (int64_t)S.sl[k];
        }
        for (size_t l = 1; l < nlen; l++)
          for (size_t k = 0; k < n; k++) {
            S.ao[l * n + k] = S.ao[k] + (int64_t)l * total;
            S.co[l * n + k] = S.co[k] + (int64_t)l * total;
          }
        if (total * (int64_t)nlen > S.floats) {
          if (S.image) prib_host_free(S.image);
          S.floats = total * (int64_t)nlen + total * (int64_t)nlen / 8;
          S.image = (float *)prib_host_alloc(sizeof(float) * (size_t)std::max<int64_t>(S.floats, 1));
          if (!S.image) fail_w(prib_last_error());
        }
        if (prib_acc_run(ctx, (int32_t)n, sp.data(), S.sl.data(), S.image, S.ao.data(), S.co.data()) != PRIB_OK)
          fail_w(prib_last_error());
        S.writing = std::async(std::launch::async, [&, k0, n, total, cur]() {
          Slot &W = slot[cur];
          std::vector<char> rec;
          for (size_t k = 0; k < n; k++) {
            const size_t q = (size_t)order[k0 + k];
            for (size_t l = 0; l < nlen; l++) {
              const int64_t bytes = rec_off[l][q + 1] - rec_off[l][q];
              rec.resize((size_t)bytes);
              prib_acc_write_record(W.image + W.ao[l * n + k], W.image + W.co[l * n + k], W.sl[k], lengths[l], rec.data());
              if (pwrite(fds[l], rec.data(), (size_t)bytes, (off_t)rec_off[l][q]) != (ssize_t)bytes) return false;
            }
          }
          __atomic_fetch_add(&sh->nt_done, total / 2, __ATOMIC_SEQ_CST);
          __atomic_fetch_add(&sh->done_chunks, 1, __ATOMIC_SEQ_CST);
          return true;
        });
        ++mine;
      }
      for (Slot &S : slot)
        if (S.writing.valid() && !S.writing.get()) fail_w("short write on an .acc file");
      for (int fd : fds) close(fd);
      if (wt.on) std::fprintf(stderr, "[db]   worker on GPU %s: %d of %d chunks\n", devs[(size_t)d].c_str(), mine, nchunks);
      wt.lap("  worker: prib_acc_run + records -> .acc");
      if (seq_ind.valid()) {
        if (!seq_ind.get()) fail_w(err_si);
        __atomic_store_n(&sh->sa_done, 1, __ATOMIC_SEQ_CST);
      }
      // no teardown: the parent stops waiting as soon as the counters say everything is on disk; freeing the DP state
      // of a CUDA context takes longer than the process exit that frees it anyway
      _exit(0);
    };

    // Demand-driven recruitment of GPUs.  Bringing up a CUDA context costs about a second per process on an NVSwitch
    // box, and start-ups of different processes do not overlap (measured: profiles/r2/db_scaling.txt), so a second
    // GPU only pays if the work still unclaimed outlasts one more start-up.  Worker 0 starts at once; worker k + 1 is
    // forked when all k + 1 running workers are up and, at the rate MEASURED so far, the unclaimed chunks would keep
    // them busy longer than the MEASURED start-up of the last context.  No model constants.
    std::vector<pid_t> workers;
    auto spawn = [&](int d) {
      const pid_t pid = fork();
      if (pid < 0) return false;
      if (pid == 0) worker_main(d);
      workers.push_back(pid);
      return true;
    };
    double t_spawn_last = since_start();
    if (!spawn(0)) return die("Error: fork failed");
    if (fixed_gpus > 0)
      for (int d = 1; d < (int)devs.size(); d++) spawn(d);
    // .nam / .bas meanwhile
    if (!write_nam_bas(err)) ok = false;
    int64_t total_nt = 0;
    for (auto &sq : seqs) total_nt += (int64_t)sq.size();
    for (;;) {
      if (__atomic_load_n(&sh->failed, __ATOMIC_SEQ_CST)) {
        workers_ok = false;
        break;
      }
      const int done = __atomic_load_n(&sh->done_chunks, __ATOMIC_SEQ_CST);
      if (done >= nchunks && __atomic_load_n(&sh->sa_done, __ATOMIC_SEQ_CST)) break;
      // a worker that died without setting the flag (killed, out of memory)
      for (pid_t pid : workers) {
        int st = 0;
        if (waitpid(pid, &st, WNOHANG) == pid && !(WIFEXITED(st) && WEXITSTATUS(st) == 0)) workers_ok = false;
      }
      if (!workers_ok) break;
      const int ready = __atomic_load_n(&sh->ready, __ATOMIC_SEQ_CST);
      if (fixed_gpus == 0 && ready == (int)workers.size() && workers.size() < devs.size()) {
        const double t_init = sh->t_last_ready - t_spawn_last;  // measured start-up of the newest worker
        const int claimed = std::min(__atomic_load_n(&sh->next_chunk, __ATOMIC_SEQ_CST), nchunks);
        const long long nt_done = __atomic_load_n(&sh->nt_done, __ATOMIC_SEQ_CST);
        const double busy = since_start() - sh->t_first_ready;
        // rate of the running workers together; before the first chunk is back, assume the rest takes forever
        const double rate = (nt_done > 0 && busy > 0) ? (double)nt_done / busy : 0.0;
        const double unclaimed_nt = (double)total_nt * (double)(nchunks - claimed) / (double)std::max(nchunks, 1);
        const double remaining = rate > 0 ? unclaimed_nt / rate : 1e30;
        if (nchunks - claimed > (int)workers.size() && remaining > t_init) {
          t_spawn_last = since_start();
          if (timer.on)
            std::fprintf(stderr, "[db] t=%.2f s: recruiting GPU %s (start-up %.2f s measured, %.2f s of work unclaimed)\n",
                         t_spawn_last, devs[workers.size()].c_str(), t_init, remaining > 1e29 ? -1.0 : remaining);
          spawn((int)workers.size());
        }
      }
      usleep(2000);
    }
    if (timer.on) std::fprintf(stderr, "[db] used %d GPU(s), one worker process each\n", (int)workers.size());
    // whoever still runs is starting up or tearing down and has nothing left to do
    for (pid_t pid : workers) {
      int st = 0;
      if (waitpid(pid, &st, WNOHANG) == 0) kill(pid, SIGKILL);
    }
    munmap(sh, 4096);
  } else {
    std::string err_si;
    if (!write_seq_ind(dbs[0], seqs, prm, err_si, nullptr) || !write_copies(err_si)) {  // test switch: host suffix arrays, no GPU
      ok = false;
      err = err_si;
    }
    if (ok && !write_nam_bas(err)) ok = false;
  }
  timer.lap("accessibility (GPU workers) + .acc/.seq/.ind");
  if (!workers_ok) return die("Error: an accessibility worker failed (see above); the database is incomplete");
  if (!ok) return die(err);
  return 0;
}
