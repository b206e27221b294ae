// rc_labels.h -- host relabelling and upload of label vectors shared by rc_post.cu and rc_predict.cu (internal).
#pragma once
#include <vector>
#include <thread>
#include <atomic>
#include <algorithm>
#include "rc_common.cuh"

// first-appearance relabelling of host label vectors to 1..K (sortlabels, utils.jl:69-74) as bytes.  Samples are
// independent: they are split over host threads.  Labels in a narrow range (the usual 1..K) go through a direct
// table, anything else through a sort.
static int compact_one(const int64_t* l, int64_t n, uint8_t* out, int* Kout, std::vector<int>& table,
                       std::vector<std::pair<int64_t, int64_t>>& tmp) {
  int64_t lo = l[0], hi = l[0];
  for (int64_t x = 1; x < n; ++x) { lo = std::min(lo, l[x]); hi = std::max(hi, l[x]); }
  if (hi - lo < (int64_t)1 << 20) {
    table.assign((size_t)(hi - lo + 1), 0);
    int K = 0;
    for (int64_t x = 0; x < n; ++x) {
      int& id = table[(size_t)(l[x] - lo)];
      if (!id) { if (K == 255) return -1; id = ++K; }
      out[x] = (uint8_t)id;
    }
    *Kout = K;
    return 0;
  }
  tmp.resize((size_t)n);
  for (int64_t x = 0; x < n; ++x) tmp[x] = {l[x], x};
  std::sort(tmp.begin(), tmp.end());
  std::vector<std::pair<int64_t, int64_t>> firsts;     // (first position, label)
  for (int64_t x = 0; x < n; ++x) if (x == 0 || tmp[x].first != tmp[x - 1].first) firsts.push_back({tmp[x].second, tmp[x].first});
  std::sort(firsts.begin(), firsts.end());
  if (firsts.size() > 255) return -1;
  *Kout = (int)firsts.size();
  std::vector<std::pair<int64_t, int>> map;             // label -> id
  for (size_t q = 0; q < firsts.size(); ++q) map.push_back({firsts[q].second, (int)q + 1});
  std::sort(map.begin(), map.end());
  for (int64_t x = 0; x < n; ++x) out[x] = (uint8_t)std::lower_bound(map.begin(), map.end(), std::make_pair(l[x], 0))->second;
  return 0;
}

static int compact_labels(const int64_t* labels, int64_t S, int64_t n, std::vector<uint8_t>& out, std::vector<int>& K) {
  out.resize((size_t)S * n); K.resize((size_t)S);
  const int64_t work = S * n;
  const int nthr = (int)std::max<int64_t>(1, std::min<int64_t>({(int64_t)std::thread::hardware_concurrency(), (int64_t)16, work / (1 << 20), S}));
  std::atomic<int64_t> bad(-1);
  auto body = [&](int w) {
    std::vector<int> table; std::vector<std::pair<int64_t, int64_t>> tmp;
    for (int64_t s = w; s < S; s += nthr)
      if (compact_one(labels + s * n, n, out.data() + s * n, &K[s], table, tmp)) { int64_t e = -1; bad.compare_exchange_strong(e, s); }
  };
  std::vector<std::thread> pool;
  for (int w = 1; w < nthr; ++w) pool.emplace_back(body, w);
  body(0);
  for (auto& t : pool) t.join();
  if (bad.load() >= 0) { rc_set_error("more than 255 clusters in sample %lld", (long long)bad.load()); return RC_ERR_SLOTS; }
  return RC_OK;
}

// The device labels of the entry points that take host label vectors: compact_labels, then the S x n bytes uploaded to
// *dL, a buffer of B.  K: every sample's number of clusters (host).
static int upload_labels(const int64_t* labels, int64_t S, int64_t n, Bufs& B, uint8_t** dL, std::vector<int>& K) {
  std::vector<uint8_t> L;
  TRYP(compact_labels(labels, S, n, L, K));
  TRYP(B.get(dL, L.size()));
  RC_CUDA(cudaMemcpy(*dL, L.data(), L.size(), cudaMemcpyHostToDevice));
  return RC_OK;
}
