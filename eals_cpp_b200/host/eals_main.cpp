// eals_main.cpp — command-line driver over the drop-in class (include/MF_fastALS.h).
//
// Does what the reference's main.cpp does (main.cpp:73-234) with the same defaults
// (main.cpp:133-144) and the same stdout lines, so transcripts diff against Outputs.txt:
//   1. read "user item score timestamp" lines; user ids are contiguous and ascending from 0
//      (main.cpp:96-112);
//   2. per user std::sort by timestamp with a plain `<` comparator — UNSTABLE, and the tie order of
//      libstdc++'s introsort is part of the split (main.cpp:35,122-124) — newest rating -> test;
//   3. the rest -> train, de-duplicated through a per-user ordered map, all values 1
//      (main.cpp:173-190); a test item can stay in train through an older duplicate;
//   4. build the model, run maxIter iterations, evaluate (main.cpp:227-231).
// Unlike the reference it takes real arguments:
//   eals_main [--data yelp.rating] [--factors 64] [--iters 20] [--w0 10] [--alpha 0.75] [--reg 0.01]
//             [--topk 10] [--no-loss] [--exact-eval] [--device 0] [--gpus N | --devices 0,1,..] [--online U,I]
//             [--save FILE] [--load FILE] [--recommend K [--recommend-out FILE]]
// --gpus N: shard users and items over GPUs device .. device+N-1 (eals_group: the exchange runs inside the
// library); --devices lists them explicitly — a repeated id puts several ranks on one GPU.
// --save / --load: factor checkpoint after training / instead of the random initialisation.
// --dump-split FILE: write the hold-one-out split (per user: test item, then the train items) and stop before
// the model is built — needs no GPU; the loader is checked against the reference's own binary this way.
// --recommend K: after training and evaluation, every user's top-K unseen items, one line "user item score" per
// recommended item (score with %.17g), to --recommend-out FILE (default: stdout).
// --online U,I: after training and evaluation, add the interaction (U, I) with the online update
// (updateModel, MF_fastALS.cpp:223-242) and print the prediction before and after.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

#include "MF_fastALS.h"
#include "eals_host_types.h"

using eals_b200::Rating;
using eals_b200::SparseMat;
using Model = eals_b200::MF_fastALS_T<SparseMat, Rating>;

static bool older_first(Rating a, Rating b) { return a.timestamp < b.timestamp; }

int main(int argc, char** argv) {
  std::string data = "yelp.rating";
  double w0 = 10, reg = 0.01, alpha = 0.75, init_mean = 0, init_stdev = 0.01;
  int factors = 64, maxIter = 20, topK = 10, threadNum = 1, device = 0;
  bool showProgress = false, showLoss = true, exact = false;
  int online_u = -1, online_i = -1, n_gpus = 1;
  std::vector<int> devices;
  std::string save_path, load_path, dump_split, recommend_out;
  int recommend_k = 0;
  for (int a = 1; a < argc; a++) {
    auto is = [&](const char* f) { return std::strcmp(argv[a], f) == 0; };
    auto next = [&]() -> const char* { if (a + 1 >= argc) { std::fprintf(stderr, "missing value after %s\n", argv[a]); std::exit(2); } return argv[++a]; };
    if (is("--data")) data = next();
    else if (is("--factors")) factors = std::atoi(next());
    else if (is("--iters")) maxIter = std::atoi(next());
    else if (is("--w0")) w0 = std::atof(next());
    else if (is("--alpha")) alpha = std::atof(next());
    else if (is("--reg")) reg = std::atof(next());
    else if (is("--topk")) topK = std::atoi(next());
    else if (is("--device")) device = std::atoi(next());
    else if (is("--gpus")) n_gpus = std::max(1, std::atoi(next()));
    else if (is("--devices")) { std::istringstream in(next()); for (std::string t; std::getline(in, t, ',');) devices.push_back(std::atoi(t.c_str())); }
    else if (is("--save")) save_path = next();
    else if (is("--load")) load_path = next();
    else if (is("--dump-split")) dump_split = next();
    else if (is("--recommend")) recommend_k = std::atoi(next());
    else if (is("--recommend-out")) recommend_out = next();
    else if (is("--no-loss")) showLoss = false;
    else if (is("--exact-eval")) exact = true;
    else if (is("--online")) { if (std::sscanf(next(), "%d,%d", &online_u, &online_i) != 2) { std::fprintf(stderr, "--online wants U,I\n"); return 2; } }
    else { std::fprintf(stderr, "unknown argument %s\n", argv[a]); return 2; }
  }

  std::cout << "Holdone out splitting" << std::endl;
  std::cout << "Sort items for each user." << std::endl;
  std::clock_t start = std::clock();
  std::ifstream fin(data);
  if (!fin.is_open()) { std::fprintf(stderr, "Error: cannot open the file %s\n", data.c_str()); return EXIT_FAILURE; }
  std::vector<std::vector<Rating>> per_user;
  int userCount = 0, itemCount = 0;
  long lines = 0;
  for (std::string line; std::getline(fin, line); lines++) {
    std::istringstream in(line);
    Rating r;
    in >> r.userId >> r.itemId >> r.score >> r.timestamp;
    if ((int)per_user.size() < r.userId + 1) per_user.emplace_back();   // one new user at a time (main.cpp:106-109)
    per_user.at(r.userId).push_back(r);
    userCount = std::max(userCount, r.userId);
    itemCount = std::max(itemCount, r.itemId);
  }
  std::cout << "line num of yelp: " << lines << std::endl;
  userCount++; itemCount++;
  if (userCount != (int)per_user.size()) { std::fprintf(stderr, "user ids must be contiguous from 0\n"); return EXIT_FAILURE; }
  for (auto& v : per_user) std::sort(v.begin(), v.end(), older_first);
  std::cout << "Sorting time:" << (double)(std::clock() - start) / CLOCKS_PER_SEC << std::endl;

  std::cout << "Generate rating matrices" << std::endl;
  start = std::clock();
  std::vector<Rating> testRatings;
  std::vector<std::map<int, double>> by_user((size_t)userCount);
  long dropped = 0;
  for (int u = 0; u < userCount; u++) {
    const auto& v = per_user[u];
    for (int i = (int)v.size() - 1; i >= 0; i--) {
      if (i == (int)v.size() - 1) testRatings.push_back(v[i]);
      else by_user[v[i].userId].insert({v[i].itemId, 1.0});
    }
    dropped += (long)v.size() - 1 - (long)by_user[u].size();
  }
  SparseMat trainMatrix(userCount, itemCount, by_user);
  std::cout << "Num of elements: " << dropped << std::endl;
  std::cout << "Generated splitted matrices time:" << (double)(std::clock() - start) / CLOCKS_PER_SEC << std::endl;
  std::cout << "Data\t" << data << std::endl;
  std::cout << "#Users\t" << userCount << std::endl;
  std::cout << "#items\t" << itemCount << std::endl;
  std::cout << "#Ratings\t" << trainMatrix.itemCount() << "\t" << "tests\t" << testRatings.size() << std::endl;
  std::cout << "==========================================" << std::endl;
  if ((int)testRatings.size() != userCount) { std::fprintf(stderr, "every user needs at least one rating\n"); return EXIT_FAILURE; }
  if (!dump_split.empty()) {
    std::ofstream out(dump_split);
    out << userCount << " " << itemCount << "\n";
    for (int u = 0; u < userCount; u++) {
      out << testRatings[u].itemId;
      for (const auto& kv : by_user[u]) out << " " << kv.first;
      out << "\n";
    }
    return out.good() ? 0 : EXIT_FAILURE;
  }

  try {
    if (!devices.empty()) n_gpus = (int)devices.size();
    Model fals(trainMatrix, testRatings, topK, threadNum, factors, maxIter, w0, alpha, reg, init_mean,
               init_stdev, showProgress, showLoss, userCount, itemCount, device, n_gpus,
               devices.empty() ? nullptr : devices.data());
    if (!load_path.empty()) fals.load(load_path);
    std::cout << "Start building model" << std::endl;
    fals.buildModel();
    if (!save_path.empty()) fals.save(save_path);
    if (n_gpus > 1) std::cerr << "replicas consistent: " << (fals.replicas_consistent() ? "yes" : "NO") << std::endl;
    std::vector<double> res = fals.evaluate(exact);
    std::cout << "<hr, ndcg, prec>: \t" << res[0] << "\t" << res[1] << "\t" << res[2] << std::endl;
    if (recommend_k > 0) {
      std::vector<int> all((size_t)userCount);
      for (int u = 0; u < userCount; u++) all[(size_t)u] = u;
      const auto rec = fals.recommend(all, recommend_k, true);
      FILE* f = recommend_out.empty() ? stdout : std::fopen(recommend_out.c_str(), "w");
      if (!f) { std::fprintf(stderr, "Error: cannot write %s\n", recommend_out.c_str()); return EXIT_FAILURE; }
      for (int u = 0; u < userCount; u++)
        for (int j = 0; j < recommend_k; j++) {
          const size_t q = (size_t)u * recommend_k + j;
          if (rec.items[q] >= 0) std::fprintf(f, "%d %d %.17g\n", u, rec.items[q], rec.scores[q]);
        }
      if (f != stdout && std::fclose(f) != 0) { std::fprintf(stderr, "Error: writing %s failed\n", recommend_out.c_str()); return EXIT_FAILURE; }
    }
    if (online_u >= 0) {
      const double before = fals.predict(online_u, online_i);
      fals.updateModel(online_u, online_i);
      std::cout.precision(17);
      std::cout << "online (" << online_u << "," << online_i << "): predict " << before << " -> "
                << fals.predict(online_u, online_i) << " loss:" << fals.loss() << std::endl;
    }
  } catch (const std::exception& e) {
    std::fprintf(stderr, "eals_main: %s\n", e.what());
    return 1;
  }
  return 0;
}
