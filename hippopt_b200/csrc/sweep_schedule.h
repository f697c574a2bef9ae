// sweep_schedule.h -- host-side list scheduler of the packed tangent sweep (kino_kin.cu).  Plain C++ (no CUDA):
// included by api.cu and compiled on its own by the CPU tests (hb_debug_sweep_schedule).
//
// Direction d (0..3 base quaternion, 4 + j joint j; SweepTopo::n_base says how many of the four quaternion
// directions take part) only needs the bodies of its sub-tree (non-zero state
// tangents: "in") and the ancestors of its joint (pure propagation of the adjoint tangent).  Those bodies are cut
// into chains that walk from a leaf towards the root; a chain ends where it meets a body that another chain of the
// same direction continues through, and flushes its running adjoint into that body's slot.  Chains are
// list-scheduled on the 32 lanes, longest remaining path first; a task may run once every flush it reads has
// landed, and two chains never flush into the same slot in the same round (the additions into a slot therefore
// happen in a fixed order).
//
// Typed rounds (round 2): an "in" task costs ~400 fp64 operations, a propagation task ~60, but a warp pays for the
// most expensive lane of a round.  Sub-tree tasks come first in every chain, so the scheduler runs rounds that hold
// at least one of them ("heavy", filled up with whatever else is ready) while any is ready, and the remaining
// propagation tasks in LIGHT rounds that hold nothing else; `heavy_mask` tells the kernel which code path a round
// takes.  (policy 0, kept for the tests: strictly homogeneous rounds of the kind with more ready work.)
#pragma once
#include <algorithm>
#include <map>
#include <utility>
#include <vector>

namespace hb {

// task descriptor of the packed tangent sweep
enum {
  KT_L_SHIFT = 0, KT_P_SHIFT = 5, KT_D_SHIFT = 10, KT_VALID = 1 << 15, KT_START = 1 << 16, KT_IN_L = 1 << 17,
  KT_IN_P = 1 << 18, KT_LOAD_SHIFT = 19, KT_FLUSH_SHIFT = 25, KT_STORE = 1u << 31  // slot ids are stored + 1 (0: none)
};

struct SweepTopo {
  int nb = 0;
  int parent[32];
  int foot_body[2];
  int chest_body = 0;
  unsigned sub_mask[32];  // bit l: body l is in the sub-tree rooted at this body
  int n_base = 4;         // base quaternion directions 0 .. n_base - 1 in the sweep (the kernel's schedule: none,
                          // it fills the quaternion columns in closed form)
};

struct SweepSchedule {
  std::vector<int> tasks;  // [round][32]
  int n_rounds = 0, n_slots = 0, n_tasks = 0, n_heavy_tasks = 0;
  unsigned seed_mask = 0;   // bit r: some task of round r sits on a foot / chest body (seed tangents needed)
  unsigned heavy_mask = 0;  // bit r: round r holds "in" tasks (full tangent arithmetic); else propagation only
  int root_slot[32] = {0};
};

inline SweepSchedule build_sweep_schedule(const SweepTopo& C, bool typed_rounds = true, int policy = 1) {
  const int nb = C.nb, n_dir = 4 + (nb - 1);
  struct Seg {
    int d;
    std::vector<int> bodies;  // leaf -> root order
    int flush_body;           // body whose slot receives the chain's state (0: the root slot; -1: the root chain)
    int crit = 0, lane = -1, next = 0, flushed = -1;
    std::vector<int> round_of;
  };
  std::vector<Seg> segs;
  std::vector<std::vector<int>> slot_of(n_dir, std::vector<int>(nb, -1));
  std::vector<std::vector<char>> in_full(n_dir, std::vector<char>(nb, 0));
  int n_slots = 0;
  for (int d = 0; d < n_dir; ++d) {
    if (d < 4 && d >= C.n_base) continue;  // a direction left out keeps no task and no slot (root_slot -1)
    const int ld = d < 4 ? 0 : d - 3;
    std::vector<char> rel(nb, 0);
    for (int l = 0; l < nb; ++l)
      if ((C.sub_mask[ld] >> l) & 1u) in_full[d][l] = rel[l] = 1;
    for (int a = C.parent[ld]; a >= 0; a = C.parent[a]) rel[a] = 1;
    // the feet-distance row couples the feet: a direction that moves one foot changes the seed applied on the
    // other, whose tangent then travels up the other leg
    for (int f = 0; f < 2; ++f)
      if (in_full[d][C.foot_body[f]])
        for (int a = C.foot_body[1 - f]; a >= 0; a = C.parent[a]) rel[a] = 1;
    // longest relevant chain below every body -> main child
    std::vector<int> height(nb, 0), main_child(nb, -1);
    for (int l = nb - 1; l >= 1; --l) {
      if (!rel[l]) continue;
      const int p = C.parent[l];
      if (rel[p] && height[l] + 1 > height[p]) {
        height[p] = height[l] + 1;
        main_child[p] = l;
      }
    }
    slot_of[d][0] = n_slots++;  // the root slot doubles as the direction's result
    for (int l = nb - 1; l >= 1; --l) {
      if (!rel[l]) continue;
      bool leaf = true;
      for (int c = l + 1; c < nb; ++c)
        if (rel[c] && C.parent[c] == l) leaf = false;
      if (!leaf) continue;
      Seg s;
      s.d = d;
      int b = l;
      for (;;) {
        s.bodies.push_back(b);
        const int p = C.parent[b];
        if (p == 0 || main_child[p] != b) {
          s.flush_body = p;
          break;
        }
        b = p;
      }
      if (s.flush_body != 0 && slot_of[d][s.flush_body] < 0) slot_of[d][s.flush_body] = n_slots++;
      segs.push_back(s);
    }
    Seg root;
    root.d = d;
    root.bodies.push_back(0);
    root.flush_body = -1;
    segs.push_back(root);
  }
  const int ns = (int)segs.size();
  // dependencies: (position inside the consumer, producer segment)
  std::vector<std::vector<std::pair<int, int>>> dep(ns);
  std::vector<int> consumer(ns, -1), consumer_pos(ns, 0);
  for (int i = 0; i < ns; ++i)
    for (int j = 0; j < ns; ++j) {
      if (i == j || segs[i].d != segs[j].d || segs[j].flush_body < 0) continue;
      for (size_t pos = 0; pos < segs[i].bodies.size(); ++pos)
        if (segs[i].bodies[pos] == segs[j].flush_body) {
          dep[i].push_back({(int)pos, j});
          consumer[j] = i;
          consumer_pos[j] = (int)pos;
        }
    }
  // critical path (segments are created leaf-first per direction, consumers may come later: iterate to a fixpoint)
  for (int i = 0; i < ns; ++i) segs[i].crit = (int)segs[i].bodies.size();
  for (int it = 0; it < nb; ++it)
    for (int j = 0; j < ns; ++j)
      if (consumer[j] >= 0) {
        const int v = (int)segs[j].bodies.size() + segs[consumer[j]].crit - consumer_pos[j];
        if (v > segs[j].crit) segs[j].crit = v;
      }
  std::vector<int> order(ns);
  for (int i = 0; i < ns; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return segs[a].crit > segs[b].crit; });
  for (Seg& s : segs) s.round_of.assign(s.bodies.size(), -1);

  auto heavy_task = [&](const Seg& s, int pos) { return in_full[s.d][s.bodies[pos]] != 0; };
  auto deps_ready = [&](int si, int pos, int r) {
    for (auto& pj : dep[si])
      if (pj.first == pos && (segs[pj.second].flushed < 0 || segs[pj.second].flushed >= r)) return false;
    return true;
  };
  std::vector<int> lane_owner(32, -1);
  std::map<std::pair<int, int>, std::vector<int>> flush_rounds;  // (direction, body) -> rounds in which it is flushed
  int remaining = ns, n_rounds = 0;
  unsigned heavy_mask = 0;
  SweepSchedule out;
  for (int r = 0; remaining > 0 && r < 32; ++r) {
    // candidates of this round: the next task of every running chain, and the first task of every chain that
    // could start (a free lane is assigned below)
    int n_free = 0;
    for (int L = 0; L < 32; ++L) n_free += lane_owner[L] < 0;
    int cnt[2] = {0, 0};  // ready tasks by kind (0 light, 1 heavy)
    {
      int free_left[2] = {n_free, n_free};
      for (int oi = 0; oi < ns; ++oi) {
        const int si = order[oi];
        Seg& s = segs[si];
        if (s.next >= (int)s.bodies.size() || !deps_ready(si, s.next, r)) continue;
        const int kind = heavy_task(s, s.next) ? 1 : 0;
        if (s.lane >= 0) ++cnt[kind];
        else if (free_left[kind] > 0) {
          ++cnt[kind];
          --free_left[kind];
        }
      }
    }
    int kind;
    if (!typed_rounds) kind = -1;
    else if (cnt[0] == 0 && cnt[1] == 0) break;  // deadlock: reported below
    else if (policy == 0) kind = cnt[1] >= cnt[0] ? 1 : 0;  // the kind with more ready work; ties: heavy
    else kind = cnt[1] > 0 ? -1 : 0;  // a round with a sub-tree task costs the full arithmetic whatever else it holds:
                                      // fill it with every ready task of either kind; otherwise a light round
    bool any = false, any_heavy = false;
    std::vector<int> release;
    // two passes over the chains in priority order: sub-tree tasks first, so that a propagation task never takes
    // the lane a sub-tree chain could have started on
    for (int pass = 0; pass < 2; ++pass)
    for (int oi = 0; oi < ns; ++oi) {
      const int si = order[oi];
      Seg& s = segs[si];
      if (s.next >= (int)s.bodies.size() || !deps_ready(si, s.next, r)) continue;
      if (s.round_of[s.next > 0 ? s.next - 1 : 0] == r && s.next > 0) continue;  // already advanced in this round
      const bool hv = heavy_task(s, s.next);
      if ((int)hv != 1 - pass) continue;
      if (kind >= 0 && (int)hv != kind) continue;
      const bool last = s.next + 1 == (int)s.bodies.size();
      if (last && s.flush_body >= 0) {
        auto& used = flush_rounds[{s.d, s.flush_body}];
        if (std::find(used.begin(), used.end(), r) != used.end()) continue;  // another chain flushes there now
      }
      if (s.lane < 0) {
        int lane = -1;
        for (int L = 0; L < 32; ++L)
          if (lane_owner[L] < 0) {
            lane = L;
            break;
          }
        if (lane < 0) continue;
        s.lane = lane;
        lane_owner[lane] = si;
      }
      if (last && s.flush_body >= 0) flush_rounds[{s.d, s.flush_body}].push_back(r);
      s.round_of[s.next] = r;
      any = true;
      any_heavy |= hv;
      ++s.next;
      if (last) {
        s.flushed = r;
        release.push_back(s.lane);  // the lane is free from the NEXT round on
        --remaining;
      }
    }
    for (int L : release) lane_owner[L] = -1;
    if (!any) break;
    if (any_heavy) heavy_mask |= 1u << r;
    n_rounds = r + 1;
  }
  if (remaining > 0) return out;  // n_rounds = 0: the caller reports the failure
  out.tasks.assign((size_t)n_rounds * 32, 0);
  for (const Seg& s : segs)
    for (size_t pos = 0; pos < s.bodies.size(); ++pos) {
      const int l = s.bodies[pos], r = s.round_of[pos];
      const int p = l == 0 ? 31 : C.parent[l];
      unsigned t = (unsigned)l << KT_L_SHIFT | (unsigned)p << KT_P_SHIFT | (unsigned)s.d << KT_D_SHIFT | KT_VALID;
      if (pos == 0) t |= KT_START;
      if (in_full[s.d][l]) t |= KT_IN_L;
      if (l != 0 && in_full[s.d][p]) t |= KT_IN_P;
      if (slot_of[s.d][l] >= 0) t |= (unsigned)(slot_of[s.d][l] + 1) << KT_LOAD_SHIFT;
      if (pos + 1 == s.bodies.size()) {
        if (l == 0) t |= (unsigned)(slot_of[s.d][0] + 1) << KT_FLUSH_SHIFT | KT_STORE;
        else t |= (unsigned)(slot_of[s.d][s.flush_body] + 1) << KT_FLUSH_SHIFT;
      }
      int& cell = out.tasks[(size_t)r * 32 + s.lane];
      if (cell != 0) {  // lane conflict: give up (n_rounds = 0)
        out.tasks.clear();
        return SweepSchedule();
      }
      cell = (int)t;
      ++out.n_tasks;
      out.n_heavy_tasks += in_full[s.d][l] ? 1 : 0;
      if (l == C.foot_body[0] || l == C.foot_body[1] || l == C.chest_body) out.seed_mask |= 1u << r;
    }
  out.n_rounds = n_rounds;
  out.n_slots = n_slots;
  out.heavy_mask = typed_rounds ? heavy_mask : 0xffffffffu;
  for (int d = 0; d < n_dir && d < 32; ++d) out.root_slot[d] = slot_of[d][0];  // -1: direction left out
  return out;
}

}  // namespace hb
