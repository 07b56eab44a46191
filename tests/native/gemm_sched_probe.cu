// Host-side probe of the persistent GEMMs' work deal (pg::make_sched / pg::next_item, csrc/gemm_persist.cuh): the same
// inline functions the kernels run, compiled for the CPU, dealt out to every CTA (pair) of a launch and checked.
//
//   gemm_sched_probe sweep   every PAIR in {1, 2}, G in [1, 148 / PAIR], N in {256, 512, 768, 1024}, the store problem
//                            alone, the split-K problem alone and both, at the live sizes around every tile and k-block
//                            edge up to 4096 and at the large sizes the plans use; prints one JSON summary line
//   gemm_sched_probe flags   one case per input line "PAIR G nprob ovh red0 N0 M0 K0 red1 N1 M1 K1"; prints one JSON
//                            line per case: whether the deal is correct and which branches of make_sched it took
//
// For every case: each (problem, tile, k-block) is dealt exactly once, no split-K item is longer than kMaxKbPerItem or
// crosses a tile, and every store item covers the tile's whole live K.
//
// The branch flags need two intermediates of make_sched (T and x_hi before its clamps); `branches` recomputes them with
// the same arithmetic and checks the recomputation against the share make_sched gave CTA 0.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../computational-chemistry-ai_b200/csrc/gemm_persist.cuh"

using namespace eims::pg;

struct Case {
  int pair, G, nprob, ovh, red[2], N[2], M[2], K[2];
};

struct Flags {
  bool split = false;       // a split-K problem is present (the balancing code runs)
  bool r_zero = false;      // r == 0: the store tiles divide evenly over the CTAs
  bool r_pos = false;       // r > 0
  bool xhi_clamped = false; // x_hi < 0 before the clamp to 0
  bool clamp_u = false;     // r * x_hi > U: the second clamp (never taken: T <= (U + r(t+1)cost + (G-r)t cost) / G)
  bool u_lt_g = false;      // fewer split-K units than CTAs: some CTAs get none
  bool multi_item = false;  // some CTA's unit range is cut into several items
  bool recompute_ok = true; // the recomputed x_hi gives CTA 0 the share make_sched gave it
};

static SchedIn sched_in(const Case& cs) {
  SchedIn in;
  in.nprob = cs.nprob; in.ovh = cs.ovh;
  for (int k = 0; k < 2; ++k) { in.red[k] = cs.red[k]; in.N[k] = cs.N[k]; }
  return in;
}

static Sched sched_of(const Case& cs, int c) {
  const SchedIn in = sched_in(cs);
  const int Mv[2] = {cs.M[0], cs.M[1]}, Kv[2] = {cs.K[0], cs.K[1]};
  return cs.pair == 2 ? make_sched<2>(in, Mv, Kv, c, cs.G) : make_sched<1>(in, Mv, Kv, c, cs.G);
}

static bool next_of(const Case& cs, const Sched& s, Cursor& cur, Item& it) {
  return cs.pair == 2 ? next_item<2>(s, cur, it) : next_item<1>(s, cur, it);
}

static Flags branches(const Case& cs) {
  Flags f;
  const Sched s0 = sched_of(cs, 0);
  if (s0.pk < 0) return f;
  f.split = true;
  const int TM = BM * cs.pair;
  const int U = ((cs.M[s0.pk] + TM - 1) / TM) * s0.nt_k * s0.KB;
  const int t = s0.tiles_s / cs.G, r = s0.tiles_s % cs.G, cost = s0.kb_s + cs.ovh;
  const int T = (U + r * (t + 1) * cost + (cs.G - r) * t * cost) / cs.G;
  int x_hi = T - (t + 1) * cost;
  f.r_zero = r == 0;
  f.r_pos = r > 0;
  f.xhi_clamped = x_hi < 0;
  if (x_hi < 0) x_hi = 0;
  f.clamp_u = r * x_hi > U;
  if (f.clamp_u) x_hi = U / (r > 0 ? r : 1);
  f.u_lt_g = U < cs.G;
  if (r > 0) f.recompute_ok = s0.u0 == 0 && s0.u1 == x_hi;
  return f;
}

// deals the whole launch; returns "" or what went wrong
static std::string check(const Case& cs, Flags* f) {
  const int TM = BM * cs.pair;
  const Sched s0 = sched_of(cs, 0);
  std::vector<int> store_cnt, unit_cnt;
  if (s0.ps >= 0) store_cnt.assign(s0.tiles_s, 0);
  if (s0.pk >= 0) unit_cnt.assign((size_t)((cs.M[s0.pk] + TM - 1) / TM) * s0.nt_k * s0.KB, 0);
  char buf[256];
  for (int c = 0; c < cs.G; ++c) {
    const Sched s = sched_of(cs, c);
    Cursor cur{0, s.u0};
    Item it;
    int items_k = 0;
    for (int guard = 0; next_of(cs, s, cur, it); ++guard) {
      if (guard > (1 << 24)) return "next_item does not terminate";
      const int pi = it.prob;
      if (pi != s.ps && pi != s.pk) return "item of an unknown problem";
      if (it.m0 % TM || it.n0 % BN || it.m0 < 0 || it.n0 < 0) return "unaligned item origin";
      if (it.m0 >= cs.M[pi] || it.n0 >= cs.N[pi]) {
        snprintf(buf, sizeof buf, "item (%d, %d) outside the live output of problem %d (CTA %d)", it.m0, it.n0, pi, c);
        return buf;
      }
      const int ntl = cs.N[pi] / BN, tile = (it.m0 / TM) * ntl + it.n0 / BN;
      if (pi == s.ps) {
        if (it.kb0 != 0 || it.nkb != s.kb_s || s.kb_s * BK < cs.K[pi]) return "store item does not cover the live K";
        ++store_cnt[tile];
      } else {
        ++items_k;
        if (it.nkb < 1 || it.nkb > kMaxKbPerItem) {
          snprintf(buf, sizeof buf, "split-K item of %d k-blocks (CTA %d)", it.nkb, c);
          return buf;
        }
        if (it.kb0 < 0 || it.kb0 + it.nkb > s.KB) {
          snprintf(buf, sizeof buf, "split-K item [%d, %d) crosses its tile of %d k-blocks (CTA %d)", it.kb0, it.kb0 + it.nkb, s.KB, c);
          return buf;
        }
        for (int k = 0; k < it.nkb; ++k) ++unit_cnt[(size_t)tile * s.KB + it.kb0 + k];
      }
    }
    if (items_k > 1 && f) f->multi_item = true;
  }
  for (size_t i = 0; i < store_cnt.size(); ++i)
    if (store_cnt[i] != 1) {
      snprintf(buf, sizeof buf, "store tile %zu dealt %d times", i, store_cnt[i]);
      return buf;
    }
  for (size_t i = 0; i < unit_cnt.size(); ++i)
    if (unit_cnt[i] != 1) {
      snprintf(buf, sizeof buf, "split-K (tile %zu, k-block %zu) dealt %d times", i / s0.KB, i % s0.KB, unit_cnt[i]);
      return buf;
    }
  return "";
}

static void print_case(const Case& c, FILE* out) {
  fprintf(out, "[%d, %d, %d, %d, %d, %d, %d, %d, %d, %d, %d, %d]", c.pair, c.G, c.nprob, c.ovh, c.red[0], c.N[0], c.M[0], c.K[0],
          c.red[1], c.N[1], c.M[1], c.K[1]);
}

// live sizes: both sides of every `step` edge up to `lim`, and the large sizes of the plans' capacities
static std::vector<int> edges(int step, int lim) {
  std::vector<int> v;
  for (int j = 0; j * step < lim; ++j) { v.push_back(j * step + 1); v.push_back((j + 1) * step); }
  for (int x : {9471, 9472, 9473, 16900, 18943, 18944, 18945, 32768, 65535}) v.push_back(x);
  return v;
}

static int sweep() {
  long long cases = 0, failures = 0;
  long long n_split = 0, n_rzero = 0, n_rpos = 0, n_xclamp = 0, n_clamp_u = 0, n_ultg = 0, n_multi = 0, n_recompute_bad = 0;
  std::string first_failure;
  Case first_case{};
  const int kk[] = {1, 31, 32, 33, 256, 512, 513, 2048};   // K of a store problem (512: one item's limit; 2048: deep mode)
  auto run = [&](const Case& cs) {
    Flags f = branches(cs);
    const std::string err = check(cs, &f);
    ++cases;
    if (!err.empty()) {
      if (failures++ == 0) { first_failure = err; first_case = cs; }
    }
    n_split += f.split; n_rzero += f.split && f.r_zero; n_rpos += f.split && f.r_pos; n_xclamp += f.xhi_clamped;
    n_clamp_u += f.clamp_u; n_ultg += f.split && f.u_lt_g; n_multi += f.multi_item; n_recompute_bad += !f.recompute_ok;
  };
  for (int pair = 1; pair <= 2; ++pair) {
    const int TM = BM * pair;
    const std::vector<int> m_edges = edges(TM, 4096), k_edges = edges(BK, 4096);
    for (int G = 1; G <= 148 / pair; ++G) {
      for (int N = 256; N <= 1024; N += 256) {
        // the store problem alone (forward / data gradient): live rows M, static K
        for (int M : m_edges)
          for (int K : kk) run(Case{pair, G, 1, 4, {0, 0}, {N, N}, {M, 0}, {K, 0}});
        // the split-K problem alone (weight gradient): M = N output rows (and a few others), live K
        for (int Mk : {1, N - 1, N, N + 1, 4 * N})
          for (int K : k_edges) run(Case{pair, G, 1, 4, {1, 0}, {N, N}, {Mk, 0}, {K, 0}});
        // both (the grouped data + weight gradient of a layer): store rows and split-K depth are the same live atom
        // count; the store problem's K and the split-K problem's rows are the hidden width N
        std::vector<int> both = m_edges;
        both.insert(both.end(), k_edges.begin(), k_edges.end());
        for (int n : both) {
          run(Case{pair, G, 2, 4, {0, 1}, {N, N}, {n, N}, {N, n}});
          run(Case{pair, G, 2, 4, {1, 0}, {N, N}, {N, n}, {n, N}});   // problems in the other order
        }
      }
    }
  }
  printf("{\"cases\": %lld, \"failures\": %lld, \"split_cases\": %lld, \"r_zero\": %lld, \"r_pos\": %lld, \"xhi_clamped\": %lld, "
         "\"clamp_u\": %lld, \"u_lt_g\": %lld, \"multi_item\": %lld, \"recompute_mismatch\": %lld, \"first_failure\": \"%s\", "
         "\"first_failing_case\": ",
         cases, failures, n_split, n_rzero, n_rpos, n_xclamp, n_clamp_u, n_ultg, n_multi, n_recompute_bad, first_failure.c_str());
  print_case(first_case, stdout);
  printf("}\n");
  return 0;
}

static int flags() {
  Case cs;
  while (scanf("%d %d %d %d %d %d %d %d %d %d %d %d", &cs.pair, &cs.G, &cs.nprob, &cs.ovh, &cs.red[0], &cs.N[0], &cs.M[0],
               &cs.K[0], &cs.red[1], &cs.N[1], &cs.M[1], &cs.K[1]) == 12) {
    Flags f = branches(cs);
    const std::string err = check(cs, &f);
    printf("{\"case\": ");
    print_case(cs, stdout);
    printf(", \"error\": \"%s\", \"split\": %d, \"r_zero\": %d, \"r_pos\": %d, \"xhi_clamped\": %d, \"clamp_u\": %d, "
           "\"u_lt_g\": %d, \"multi_item\": %d, \"recompute_ok\": %d}\n",
           err.c_str(), f.split, f.r_zero, f.r_pos, f.xhi_clamped, f.clamp_u, f.u_lt_g, f.multi_item, f.recompute_ok);
  }
  return 0;
}

int main(int argc, char** argv) {
  if (argc == 2 && !strcmp(argv[1], "sweep")) return sweep();
  if (argc == 2 && !strcmp(argv[1], "flags")) return flags();
  fprintf(stderr, "usage: %s sweep | flags\n", argv[0]);
  return 2;
}
