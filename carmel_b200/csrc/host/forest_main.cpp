// forest_main.cpp -- `forest-em-b200`: forest-em's command line (training subset) on the GPU library.
// Mirrors ForestEmParams::main / perform_forest_em (forest-em/forest-em-params.hpp:262-293,
// forest-em-params.cpp:62-148): exit code 0 on success, 1 on any error with "ERROR: ..." on stderr.
//
//   forest-em-b200 --gpus=N ...   forests sharded over GPUs 0..N-1 of this box (one job and one host thread per GPU,
//                                 --shard=r/N --gpu=r); the rule count table is all-reduced with NCCL every iteration;
//                                 rank 0 logs and writes the outputs.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <string>
#include <thread>
#include <vector>

#include "carmel_b200.h"

static int run_multi_gpu(int argc, char** argv, int n_gpus) {
  for (int i = 1; i < argc; ++i) {
    if (std::strncmp(argv[i], "--kbest", 7) == 0) {
      std::cerr << "ERROR: --kbest decodes on one GPU (no --gpus / --shard)\n\nTry 'forest-em -h' for documentation\n";
      return 1;
    }
    if (std::strncmp(argv[i], "--sample=", 9) == 0 || std::strcmp(argv[i], "--sample") == 0) {
      std::cerr << "ERROR: --sample draws on one GPU (no --gpus / --shard)\n\nTry 'forest-em -h' for documentation\n";
      return 1;
    }
  }
  unsigned char id[CML_COMM_ID_BYTES];
  if (cml_comm_unique_id(id) != CML_OK) {
    std::cerr << "ERROR: --gpus needs NCCL (libnccl.so.2 could not be loaded)\n";
    return 1;
  }
  std::vector<cml_forest_job*> jobs(n_gpus, nullptr);
  std::vector<std::vector<std::string>> args(n_gpus);
  for (int r = 0; r < n_gpus; ++r) {
    for (int i = 0; i < argc; ++i) {
      if (std::strncmp(argv[i], "--gpus", 6) == 0 || std::strncmp(argv[i], "--gpu=", 6) == 0) continue;
      // outputs belong to rank 0 (every rank holds the same parameters; per-forest files would cover one block only)
      if (r > 0 && i > 0) {
        const char* a = argv[i];
        const bool valued = !std::strcmp(a, "-o") || !std::strcmp(a, "-O") || !std::strcmp(a, "-S") || !std::strcmp(a, "-x") ||
                            !std::strcmp(a, "--outparam-file") || !std::strcmp(a, "--outcounts-file") ||
                            !std::strcmp(a, "--out-per-forest-inside-sum") || !std::strcmp(a, "--checkpoint-prefix");
        if (valued) {
          ++i;
          continue;
        }
        if (!std::strcmp(a, "-c") || !std::strcmp(a, "--checkpoint-parameters") || !std::strncmp(a, "--history", 9) ||
            !std::strncmp(a, "--outparam-file=", 16) || !std::strncmp(a, "--outcounts-file=", 17) ||
            !std::strncmp(a, "--print-forests", 15))
          continue;
      }
      args[r].push_back(argv[i]);
    }
    args[r].push_back("--shard=" + std::to_string(r) + "/" + std::to_string(n_gpus));
    args[r].push_back("--gpu=" + std::to_string(r));
    std::vector<const char*> av;
    for (auto const& a : args[r]) av.push_back(a.c_str());
    if (cml_forest_job_open(&jobs[r], (int)av.size(), av.data()) != CML_OK) {
      for (auto* j : jobs) cml_forest_job_close(j);
      return 1;
    }
    cml_forest_job_set_comm(jobs[r], id);
    if (r > 0) cml_forest_job_set_quiet(jobs[r], 1);
  }
  std::vector<int> rcs(n_gpus, CML_OK);
  std::vector<std::thread> th;
  for (int r = 0; r < n_gpus; ++r) th.emplace_back([&, r]() { rcs[r] = cml_forest_job_train(jobs[r]); });
  for (auto& t : th) t.join();
  int rc = CML_OK;
  for (int r = 0; r < n_gpus; ++r)
    if (rcs[r] != CML_OK) {
      std::cerr << "ERROR (GPU " << r << "): " << cml_forest_job_error(jobs[r]) << "\n";
      rc = rcs[r];
    }
  if (rc == CML_OK) rc = cml_forest_job_write(jobs[0]);
  for (auto* j : jobs) cml_forest_job_close(j);
  return rc == CML_OK ? 0 : 1;
}

int main(int argc, char** argv) {
  for (int i = 1; i < argc; ++i)
    if (std::strncmp(argv[i], "--gpus=", 7) == 0 && std::atoi(argv[i] + 7) > 1) return run_multi_gpu(argc, argv, std::atoi(argv[i] + 7));
  cml_forest_job* job = nullptr;
  int rc = cml_forest_job_open(&job, argc, (const char* const*)argv);
  if (rc != CML_OK) {
    cml_forest_job_close(job);
    return 1;
  }
  rc = cml_forest_job_train(job);
  if (rc == CML_OK) rc = cml_forest_job_write(job);
  if (rc != CML_OK) std::cerr << "ERROR: " << cml_forest_job_error(job) << "\n\nTry 'forest-em -h' for documentation\n";
  cml_forest_job_close(job);
  return rc == CML_OK ? 0 : 1;
}
