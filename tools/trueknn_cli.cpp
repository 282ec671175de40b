// trueknn_cli.cpp — the sample's command line over libtrueknn (C++ host side of the drop-in).
//
//   trueknn <file> <n> <dim> <start radius> <k> <output file> [--neighbours <path> [--binary]] [--device <d>] [--json]
//           [--gpus <N> | --devices <a,b,...>] [--mode shard|partition] [--dbscan <eps> <min_pts> [--labels <path> [--binary]]]
//           [--radius-search <r> [--neighbours <path> [--binary]]]
//
// --radius-search runs the exact fixed-radius neighbour lists (tknn_radius_search) instead of the kNN search after the
// build; k and the start radius are still required and are ignored.  --neighbours then writes one
// `query,neighbourIndex,distance` line per entry, or <path>.off.u64 / .idx.i32 / .dist.f32 with --binary.
// --dbscan runs exact DBSCAN (tknn_dbscan) instead of the kNN search after the build; k and the start radius are still
// required and are ignored.  --labels writes `point,label` lines (label -1 = noise), or raw int32 labels with --binary.
// --gpus N (devices 0..N-1) or --devices (an explicit list; naming one device several times runs that many ranks on
// it) drives all devices from this one process through tknn_create_multi: the device-list form of the reference's
// owlContextCreate(ids, n) (owl/include/owl/owl_host.h:360; the sample itself passes one device, hostCode.cpp:141).
// --mode shard: BVH replicated, queries sharded; --mode partition: points partitioned by Morton range.
//
// Mirrors samples/s01-trueknn/hostCode.cpp main() (argv contract :66-73): reads the first n points of
// a text file (grammar :83-104, 2-D/3-D handling :114-124), builds the accel ("Build time",
// :201-212), runs the rounds ("True KNN time", :279-347), prints the same three lines and appends
// "Total time" to the output file (:346-356).  What the reference leaves commented out (:312-319) —
// writing `query,neighbourIndex,distance` lines — is available behind --neighbours.
// Unlike the reference it returns a non-zero exit code with a message instead of perror/exit in the
// middle of the run, and rejects k > n-1 (the reference loops forever, :285,321-323).
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "../include/trueknn.h"

int main(int ac, char** av) {
  std::vector<std::string> pos;
  std::string neigh_path, labels_path, mode = "shard";
  bool dbscan = false, radius_search = false;
  float rs_radius = 0.f;
  float db_eps = 0.f;
  int db_min_pts = 0;
  std::vector<int> devices;
  int device = 0;
  bool json = false, binary = false;
  for (int i = 1; i < ac; ++i) {
    const std::string a = av[i];
    if (a == "--neighbours" || a == "--neighbors") { if (++i < ac) neigh_path = av[i]; }
    else if (a == "--device") { if (++i < ac) device = std::atoi(av[i]); }
    else if (a == "--gpus") { if (++i < ac) { devices.clear(); for (int d = 0; d < std::atoi(av[i]); ++d) devices.push_back(d); } }
    else if (a == "--devices") {
      if (++i < ac) {
        devices.clear();
        for (const char* p = av[i]; *p;) { devices.push_back(std::atoi(p)); while (*p && *p != ',') ++p; if (*p == ',') ++p; }
      }
    }
    else if (a == "--mode") { if (++i < ac) mode = av[i]; }
    else if (a == "--dbscan") {
      dbscan = true;
      if (i + 2 < ac) { db_eps = (float)std::atof(av[i + 1]); db_min_pts = std::atoi(av[i + 2]); }
      i += 2;
    }
    else if (a == "--radius-search") { radius_search = true; if (++i < ac) rs_radius = (float)std::atof(av[i]); }
    else if (a == "--labels") { if (++i < ac) labels_path = av[i]; }
    else if (a == "--json") json = true;
    else if (a == "--binary") binary = true;  // --neighbours as raw arrays: <path>.idx.i32 / <path>.dist.f32
    else pos.push_back(a);
  }
  if (pos.size() != 6 || (mode != "shard" && mode != "partition") || ((dbscan || radius_search) && !devices.empty()) ||
      (dbscan && radius_search)) {
    std::fprintf(stderr, "usage: %s <file> <n> <dim> <start radius> <k> <output file> [--neighbours <path>] [--device <d>] [--json]\n"
                         "          [--gpus <N> | --devices <a,b,...>] [--mode shard|partition]\n"
                         "          [--dbscan <eps> <min_pts> [--labels <path> [--binary]]]   (one GPU)\n"
                         "          [--radius-search <r> [--neighbours <path> [--binary]]]   (one GPU)\n", av[0]);
    return 64;
  }
  const std::string path = pos[0], outfile = pos[5];
  const long long n = std::atoll(pos[1].c_str());
  const int dim = std::atoi(pos[2].c_str());
  const float radius = (float)std::atof(pos[3].c_str());
  const int k = std::atoi(pos[4].c_str());
  if (dim != 2 && dim != 3) { std::fprintf(stderr, "dimension must be 2 or 3\n"); return 65; }

  // grammar of hostCode.cpp:83-124 (parallel mmap parser in libtrueknn; rows come back as x, y, z with z = 0 for 2-D)
  if (n < 0) { std::fprintf(stderr, "number of points must be >= 0\n"); return 65; }
  std::vector<float> flat((size_t)(n + 8) * 3);
  uint64_t np = 0;
  int rrc = tknn_read_points(path.c_str(), (uint64_t)n, dim, flat.data(), (uint64_t)n + 8, &np);
  if (rrc == TKNN_EINVAL && np > (uint64_t)n + 8) {  // several points per line: the last line read is consumed whole
    const uint64_t cap = np;
    flat.resize((size_t)cap * 3);
    rrc = tknn_read_points(path.c_str(), (uint64_t)n, dim, flat.data(), cap, &np);
  }
  if (rrc != TKNN_OK) {
    std::fprintf(stderr, "cannot read %s as %d-D points (unreadable, or the float count is not a multiple of dim — "
                         "the reference throws std::out_of_range there)\n", path.c_str(), dim);
    return 66;
  }
  std::cout << " num spheres: " << np << "\n";

  if (!devices.empty()) {
    // ---- all devices from this process (tknn_create_multi) ----
    tknn_multi* mg = nullptr;
    int mrc = tknn_create_multi(devices.data(), (int)devices.size(), mode == "shard" ? TKNN_SHARD_QUERIES : TKNN_PARTITION_POINTS, &mg);
    if (mrc != TKNN_OK) { std::fprintf(stderr, "tknn_create_multi failed (%d): CUDA sm_100 devices and NCCL are required\n", mrc); return 70; }
    auto m0 = std::chrono::steady_clock::now();
    mrc = tknn_multi_build(mg, flat.data(), np, 3, 3);
    auto m1 = std::chrono::steady_clock::now();
    if (mrc != TKNN_OK) { std::fprintf(stderr, "tknn_multi_build: %s\n", tknn_multi_last_error(mg)); tknn_multi_destroy(mg); return 71; }
    const double mbuild_s = std::chrono::duration<double>(m1 - m0).count();
    std::cout << "Build time: " << mbuild_s << '\n';
    std::vector<int32_t> midx((size_t)np * k);
    std::vector<float> mdist((size_t)np * k);
    auto m2 = std::chrono::steady_clock::now();
    mrc = tknn_multi_search(mg, k, radius, midx.data(), mdist.data());
    auto m3 = std::chrono::steady_clock::now();
    if (mrc != TKNN_OK) { std::fprintf(stderr, "tknn_multi_search: %s\n", tknn_multi_last_error(mg)); tknn_multi_destroy(mg); return 72; }
    const double mknn_s = std::chrono::duration<double>(m3 - m2).count();
    for (int r = 0; r < tknn_multi_ranks(mg); ++r) {
      tknn_stats st;
      tknn_get_stats(tknn_multi_ctx(mg, r), &st);
      std::cout << "GPU " << devices[r] << " (rank " << r << "): " << st.n_queries << " queries, " << st.rounds << " rounds, start radius "
                << st.start_radius << ", search " << st.search_ms / 1000.0 << " seconds\n";
    }
    std::cout << "True KNN time: " << mknn_s << " seconds." << std::endl;
    std::cout << "Total time: " << mbuild_s + mknn_s << '\n';
    std::ofstream mout(outfile, std::ios::app);
    if (!mout.is_open()) { std::perror("Error open"); tknn_multi_destroy(mg); return 73; }
    mout << mbuild_s + mknn_s << std::endl;
    if (!neigh_path.empty() && tknn_write_neighbours(neigh_path.c_str(), midx.data(), mdist.data(), np, k, binary ? 1 : 0) != TKNN_OK) {
      std::perror("Error open");
      tknn_multi_destroy(mg);
      return 73;
    }
    if (json) {
      float tm[4];
      tknn_multi_get_times(mg, tm);
      std::printf("{\"n\": %llu, \"k\": %d, \"gpus\": %d, \"mode\": \"%s\", \"build_ms\": %.4f, \"search_ms\": %.4f, "
                  "\"exchange_ms\": %.4f, \"d2h_ms\": %.4f}\n",
                  (unsigned long long)np, k, (int)devices.size(), mode.c_str(), tm[0], tm[1], tm[2], tm[3]);
    }
    tknn_multi_destroy(mg);
    return 0;
  }

  tknn_ctx* ctx = nullptr;
  int rc = tknn_create(device, &ctx);
  if (rc != TKNN_OK) { std::fprintf(stderr, "tknn_create failed (%d): a CUDA sm_100 device is required\n", rc); return 70; }

  auto t0 = std::chrono::steady_clock::now();
  rc = tknn_build(ctx, flat.data(), np, 3, 3);
  auto t1 = std::chrono::steady_clock::now();
  if (rc != TKNN_OK) { std::fprintf(stderr, "tknn_build: %s\n", tknn_last_error(ctx)); tknn_destroy(ctx); return 71; }
  const double build_s = std::chrono::duration<double>(t1 - t0).count();
  std::cout << "Build time: " << build_s << '\n';

  if (dbscan) {
    std::vector<int32_t> labels((size_t)np);
    uint64_t n_clusters = 0;
    auto d0 = std::chrono::steady_clock::now();
    rc = tknn_dbscan(ctx, db_eps, db_min_pts, labels.data(), nullptr, &n_clusters);
    auto d1 = std::chrono::steady_clock::now();
    if (rc != TKNN_OK) { std::fprintf(stderr, "tknn_dbscan: %s\n", tknn_last_error(ctx)); tknn_destroy(ctx); return 72; }
    const double db_s = std::chrono::duration<double>(d1 - d0).count();
    tknn_stats st;
    tknn_get_stats(ctx, &st);
    static const char* phase[4] = {"core test", "link", "labelling", "border"};
    for (int i = 0; i < 4; ++i)
      std::cout << "Phase: " << phase[i] << " Queries = " << st.round_queries[i] << " Time: " << st.round_ms[i] / 1000.0 << " seconds\n";
    uint64_t noise = 0;
    for (int32_t l : labels) noise += l < 0;
    std::cout << "Clusters: " << n_clusters << " Noise points: " << noise << '\n';
    std::cout << "DBSCAN time: " << db_s << " seconds." << std::endl;
    const double tot = build_s + db_s;
    std::cout << "Total time: " << tot << '\n';
    std::ofstream out(outfile, std::ios::app);
    if (!out.is_open()) { std::perror("Error open"); tknn_destroy(ctx); return 73; }
    out << tot << std::endl;
    if (!labels_path.empty()) {
      FILE* f = std::fopen(labels_path.c_str(), binary ? "wb" : "w");
      bool ok = f != nullptr;
      if (ok && binary) ok = std::fwrite(labels.data(), sizeof(int32_t), labels.size(), f) == labels.size();
      for (size_t i = 0; ok && !binary && i < labels.size(); ++i) ok = std::fprintf(f, "%zu,%d\n", i, labels[i]) > 0;
      if (f && std::fclose(f) != 0) ok = false;
      if (!ok) { std::perror("Error open"); tknn_destroy(ctx); return 73; }
    }
    if (json) {
      std::printf("{\"n\": %llu, \"eps\": %.9g, \"min_pts\": %d, \"clusters\": %llu, \"noise\": %llu, \"build_ms\": %.4f, "
                  "\"dbscan_ms\": %.4f, \"points_per_s\": %.1f}\n",
                  (unsigned long long)np, db_eps, db_min_pts, (unsigned long long)n_clusters, (unsigned long long)noise, st.build_ms,
                  st.search_ms, st.search_ms > 0 ? np / (st.search_ms * 1e-3) : 0.0);
    }
    tknn_destroy(ctx);
    return 0;
  }

  if (radius_search) {
    std::vector<uint64_t> offsets((size_t)np + 1);
    uint64_t total = 0;
    auto s0 = std::chrono::steady_clock::now();
    rc = tknn_radius_search(ctx, rs_radius, offsets.data(), nullptr, nullptr, 0, &total);  // size query
    std::vector<int32_t> ridx;
    std::vector<float> rdist;
    if (rc == TKNN_OK) {
      ridx.resize((size_t)total);
      rdist.resize((size_t)total);
      rc = tknn_radius_search(ctx, rs_radius, offsets.data(), ridx.data(), rdist.data(), total, &total);
    }
    auto s1 = std::chrono::steady_clock::now();
    if (rc != TKNN_OK) { std::fprintf(stderr, "tknn_radius_search: %s\n", tknn_last_error(ctx)); tknn_destroy(ctx); return 72; }
    const double rs_s = std::chrono::duration<double>(s1 - s0).count();
    tknn_stats st;
    tknn_get_stats(ctx, &st);
    static const char* phase[3] = {"count", "fill", "order"};
    for (int i = 0; i < 3; ++i)
      std::cout << "Phase: " << phase[i] << " Queries = " << st.round_queries[i] << " Time: " << st.round_ms[i] / 1000.0 << " seconds\n";
    std::cout << "Neighbours: " << total << '\n';
    std::cout << "Radius search time: " << rs_s << " seconds." << std::endl;
    const double tot = build_s + rs_s;
    std::cout << "Total time: " << tot << '\n';
    std::ofstream out(outfile, std::ios::app);
    if (!out.is_open()) { std::perror("Error open"); tknn_destroy(ctx); return 73; }
    out << tot << std::endl;
    if (!neigh_path.empty() &&
        tknn_write_neighbour_lists(neigh_path.c_str(), offsets.data(), ridx.data(), rdist.data(), np, binary ? 1 : 0) != TKNN_OK) {
      std::perror("Error open");
      tknn_destroy(ctx);
      return 73;
    }
    if (json) {
      std::printf("{\"n\": %llu, \"radius\": %.9g, \"neighbours\": %llu, \"build_ms\": %.4f, \"radius_ms\": %.4f}\n",
                  (unsigned long long)np, rs_radius, (unsigned long long)total, st.build_ms, st.search_ms);
    }
    tknn_destroy(ctx);
    return 0;
  }

  std::vector<int32_t> idx((size_t)np * k);
  std::vector<float> dist((size_t)np * k);
  auto t2 = std::chrono::steady_clock::now();
  rc = tknn_search(ctx, k, radius, idx.data(), dist.data());
  auto t3 = std::chrono::steady_clock::now();
  if (rc != TKNN_OK) { std::fprintf(stderr, "tknn_search: %s\n", tknn_last_error(ctx)); tknn_destroy(ctx); return 72; }
  const double knn_s = std::chrono::duration<double>(t3 - t2).count();
  tknn_stats st;
  tknn_get_stats(ctx, &st);
  float r = st.start_radius;
  for (int i = 0; i < st.rounds && i < TKNN_MAX_ROUNDS; ++i, r *= 2) {
    std::cout << "Round: " << (i + 1) << " Radius = " << r << " Queries = " << st.round_queries[i]
              << " Time: " << st.round_ms[i] / 1000.0 << " seconds\n";
  }
  std::cout << "True KNN time: " << knn_s << " seconds." << std::endl;
  const double tot = build_s + knn_s;
  std::cout << "Total time: " << tot << '\n';

  std::ofstream out(outfile, std::ios::app);
  if (!out.is_open()) { std::perror("Error open"); tknn_destroy(ctx); return 73; }
  out << tot << std::endl;

  if (!neigh_path.empty()) {
    if (tknn_write_neighbours(neigh_path.c_str(), idx.data(), dist.data(), np, k, binary ? 1 : 0) != TKNN_OK) {
      std::perror("Error open");
      tknn_destroy(ctx);
      return 73;
    }
  }
  if (json) {
    std::printf("{\"n\": %llu, \"k\": %d, \"rounds\": %d, \"build_ms\": %.4f, \"search_ms\": %.4f, \"start_radius\": %.9g, "
                "\"queries_per_s\": %.1f}\n",
                (unsigned long long)np, k, st.rounds, st.build_ms, st.search_ms, st.start_radius,
                st.search_ms > 0 ? np / (st.search_ms * 1e-3) : 0.0);
  }
  tknn_destroy(ctx);
  return 0;
}
