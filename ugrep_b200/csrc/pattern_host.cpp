// pattern_host.cpp — DFA export (host).  See pattern_host.hpp.
//
// Input format: the opcode words reflex::Pattern::encode_dfa writes
// (/root/reference/lib/pattern.cpp:2823-3063; codec include/reflex/pattern.h:1155-1247):
//   state := [TAKE] META* GOTO+      (state id = index of its first word)
//   GOTO  := lo<<24 | hi<<16 | idx16 (idx 0xFFFF = HALT, 0xFFFE = LONG: next word 0xFF<<24 | idx24)
//   META  := (meta-0x100)<<24 | idx16, same LONG rule
//   TAKE  := 0xFE<<24 | accept24
// A byte is resolved by first match over the GOTO list, exactly as the interpreter's
// range search does (lib/matcher.cpp:467-502).
#include "pattern_host.hpp"

#include <algorithm>
#include <cstring>
#include <map>
#include <queue>

namespace ugx {

int select_advance(const ugx_prefilter& pf, uint32_t matcher_flags)
{
  if (pf.len == 0)
  {
    if (pf.min == 0 && (matcher_flags & UGX_OPT_N))
      return UGX_ADV_NONE;
    if (pf.pin == 1)
      return pf.min < 2 ? UGX_ADV_PIN1_ONE : pf.min < 4 ? UGX_ADV_PIN1_PMA : UGX_ADV_PIN1_PMH;
    if ((pf.pin >= 2 && pf.pin <= 8) || pf.pin == 16)
      return pf.min < 2 ? UGX_ADV_PIN_ONE : pf.min < 4 ? UGX_ADV_PIN_PMA : UGX_ADV_PIN_PMH;
    // bitap vs PM4 thresholds of the x86 SIMD builds (MAX_PATTERN_MIN{1,2,3}_NPY, lib/matcher.cpp:782-794)
    switch (pf.min)
    {
      case 0:
      case 1: return pf.npy <= 33 ? UGX_ADV_MIN1 : UGX_ADV_PMA;
      case 2: return pf.npy <= 36 ? UGX_ADV_MIN2 : UGX_ADV_PMA;
      case 3: return pf.npy <= 47 ? UGX_ADV_MIN3 : UGX_ADV_PMA;
      default: return UGX_ADV_MIN4;
    }
  }
  if (pf.len == 1)
    return pf.min == 0 ? UGX_ADV_CHAR : pf.min < 4 ? UGX_ADV_CHAR_PMA : UGX_ADV_CHAR_PMH;
  // advance_chars<2|3>, advance_string and advance_string_bm are exact literal searches that differ
  // only in how they skip; one predicate covers them
  return pf.min == 0 ? UGX_ADV_STRING : pf.min < 4 ? UGX_ADV_STRING_PMA : UGX_ADV_STRING_PMH;
}

namespace {

struct RawState {
  uint32_t accept = 0;
  std::vector<std::pair<uint32_t, uint32_t>> metas; // (code, target word)
  uint32_t target[256];                             // target word or NONE
};

constexpr uint32_t NONE = 0xFFFFFFFFu;

int parse_state(const uint32_t* opc, uint32_t nop, uint32_t s, RawState& st, std::string& err)
{
  uint32_t i = s;
  auto word = [&](uint32_t k) -> uint32_t { return k < nop ? opc[k] : OP_HALT; };
  if (s >= nop)
  {
    err = "jump outside the opcode table";
    return UGX_E_INVALID;
  }
  uint32_t op = word(i);
  if (!op_is_goto(op) && (op >> 24) == 0xfe)
  {
    st.accept = op & 0xffffff;
    op = word(++i);
  }
  while (!op_is_goto(op))
  {
    uint32_t code = op >> 24;
    if (code == 0xfd || code == 0xfc || code == 0xfb)
    {
      err = "REDO/TAIL/HEAD opcodes (lookahead, negative patterns) are outside the path's scope";
      return UGX_E_UNSUPPORTED;
    }
    if (code == 0xfe)
    {
      err = "unexpected TAKE inside a state";
      return UGX_E_INVALID;
    }
    if (code == 0xff)
    {
      op = word(++i);
      continue;
    }
    if (code == 0 || code > 0x0c)
    {
      err = "indent/dedent META opcodes are outside the path's scope";
      return UGX_E_UNSUPPORTED;
    }
    uint32_t idx = op & 0xffff;
    if (idx == IDX_LONG)
      idx = word(++i) & 0xffffff;
    else if (idx == IDX_HALT)
    {
      err = "META edge to the dead state";
      return UGX_E_INVALID;
    }
    st.metas.emplace_back(code, idx);
    op = word(++i);
    if (i > nop)
    {
      err = "unterminated state";
      return UGX_E_INVALID;
    }
  }
  const uint32_t g0 = i;
  for (uint32_t b = 0; b < 256; ++b)
  {
    uint32_t j = g0;
    uint32_t o = word(j);
    while (b < (o >> 24) || b > ((o >> 16) & 0xff))
    {
      o = word(++j);
      if (j > nop)
      {
        err = "unterminated goto list";
        return UGX_E_INVALID;
      }
    }
    uint32_t idx = o & 0xffff;
    if (idx == IDX_HALT)
      st.target[b] = NONE;
    else if (idx == IDX_LONG)
      st.target[b] = word(j + 1) & 0xffffff;
    else
      st.target[b] = idx;
  }
  return UGX_OK;
}

} // namespace

int flatten_dfa(const uint32_t* opc, uint32_t nop, HostDfa& out, std::string& err)
{
  if (opc == nullptr || nop == 0)
  {
    err = "empty opcode table";
    return UGX_E_INVALID;
  }
  std::map<uint32_t, uint32_t> id_of; // word index -> dense id (BFS order, start = 0)
  std::vector<RawState> states;
  std::vector<uint32_t> word_of;
  std::queue<uint32_t> todo;
  id_of[0] = 0;
  word_of.push_back(0);
  todo.push(0);
  while (!todo.empty())
  {
    uint32_t w = todo.front();
    todo.pop();
    RawState st;
    int rc = parse_state(opc, nop, w, st, err);
    if (rc != UGX_OK)
      return rc;
    auto visit = [&](uint32_t t) {
      if (t != NONE && id_of.find(t) == id_of.end())
      {
        id_of[t] = static_cast<uint32_t>(word_of.size());
        word_of.push_back(t);
        todo.push(t);
      }
    };
    for (uint32_t b = 0; b < 256; ++b)
      visit(st.target[b]);
    for (auto& m : st.metas)
      visit(m.second);
    if (states.size() <= id_of[w])
      states.resize(id_of[w] + 1);
    states[id_of[w]] = st;
    if (word_of.size() >= DEAD)
    {
      err = "more than 65534 DFA states";
      return UGX_E_UNSUPPORTED;
    }
  }
  const uint32_t ns = static_cast<uint32_t>(word_of.size());
  states.resize(ns);
  // renumber: 0 = start | non-accepting with byte edges | accepting with byte edges | leaves (no byte edges).
  // The scan kernels then test "accepting or leaf" with one compare against first_acc.
  {
    auto category = [&](uint32_t s) -> int {
      bool edges = false;
      for (uint32_t b = 0; b < 256 && !edges; ++b)
        edges = states[s].target[b] != NONE;
      return !edges ? 2 : states[s].accept != 0 ? 1 : 0;
    };
    std::vector<uint32_t> order; // new id -> old id
    order.push_back(0);
    uint32_t first[3] = {0, 0, 0};
    for (int cat = 0; cat < 3; ++cat)
    {
      first[cat] = static_cast<uint32_t>(order.size());
      for (uint32_t s = 1; s < ns; ++s)
        if (category(s) == cat)
          order.push_back(s);
    }
    out.first_acc = first[1];
    out.first_leaf = first[2];
    std::vector<RawState> st2(ns);
    std::vector<uint32_t> w2(ns);
    for (uint32_t i = 0; i < ns; ++i)
    {
      st2[i] = states[order[i]];
      w2[i] = word_of[order[i]];
      id_of[w2[i]] = i;
    }
    states.swap(st2);
    word_of.swap(w2);
  }
  // byte equivalence classes: bytes with identical columns
  std::map<std::vector<uint32_t>, uint32_t> col_id;
  uint32_t ncls = 0;
  std::vector<uint32_t> rep; // representative byte per class
  for (uint32_t b = 0; b < 256; ++b)
  {
    std::vector<uint32_t> col(ns);
    for (uint32_t s = 0; s < ns; ++s)
      col[s] = states[s].target[b];
    auto it = col_id.find(col);
    if (it == col_id.end())
    {
      col_id[col] = ncls;
      out.cls[b] = static_cast<uint8_t>(ncls);
      rep.push_back(b);
      ++ncls;
    }
    else
    {
      out.cls[b] = static_cast<uint8_t>(it->second);
    }
  }
  out.nstates = ns;
  out.ncls = ncls;
  out.next.assign(static_cast<size_t>(ns) * ncls, DEAD);
  out.accept.assign(ns, 0);
  out.word_of = word_of;
  out.meta_off.assign(ns + 1, 0);
  out.metas.clear();
  out.has_meta = false;
  out.newline_live = false;
  out.to_start = false;
  for (uint32_t s = 0; s < ns; ++s)
  {
    out.accept[s] = states[s].accept;
    for (uint32_t c = 0; c < ncls; ++c)
    {
      uint32_t t = states[s].target[rep[c]];
      if (t != NONE)
      {
        uint32_t id = id_of[t];
        out.next[static_cast<size_t>(s) * ncls + c] = static_cast<uint16_t>(id);
        if (id == 0)
          out.to_start = true;
      }
    }
    if (states[s].target['\n'] != NONE)
      out.newline_live = true;
    out.meta_off[s] = static_cast<uint32_t>(out.metas.size());
    for (auto& m : states[s].metas)
    {
      out.metas.push_back(MetaEdge{m.first, id_of[m.second]});
      out.has_meta = true;
    }
  }
  out.meta_off[ns] = static_cast<uint32_t>(out.metas.size());
  // longest match: longest path from the start state (byte edges weigh 1, META edges 0); a cycle makes it unbounded
  {
    std::vector<int> color(ns, 0);          // 0 new, 1 on the stack, 2 done
    std::vector<uint32_t> depth(ns, 0);     // longest path from the state
    std::vector<std::pair<uint32_t, uint32_t>> stack; // (state, next successor index)
    bool cyclic = false;
    auto succ = [&](uint32_t s, uint32_t i, uint32_t& to, uint32_t& w) -> bool {
      if (i < ncls)
      {
        const uint16_t t = out.next[static_cast<size_t>(s) * ncls + i];
        to = t;
        w = 1;
        return true;
      }
      const uint32_t m = out.meta_off[s] + (i - ncls);
      if (m < out.meta_off[s + 1])
      {
        to = out.metas[m].target;
        w = 0;
        return true;
      }
      return false;
    };
    stack.emplace_back(0u, 0u);
    color[0] = 1;
    while (!stack.empty() && !cyclic)
    {
      const uint32_t s = stack.back().first;
      uint32_t to = 0, w = 0;
      if (!succ(s, stack.back().second, to, w))
      {
        color[s] = 2;
        stack.pop_back();
        continue;
      }
      ++stack.back().second;
      if (to == DEAD)
        continue;
      if (color[to] == 1)
        cyclic = true;
      else if (color[to] == 0)
      {
        color[to] = 1;
        stack.emplace_back(to, 0u);
      }
    }
    if (cyclic)
      out.max_match_len = 0xFFFFFFFFu;
    else
    {
      // states in reverse finishing order are not kept: relax repeatedly (ns is small, the graph acyclic)
      bool changed = true;
      while (changed)
      {
        changed = false;
        for (uint32_t s = 0; s < ns; ++s)
          for (uint32_t i = 0;; ++i)
          {
            uint32_t to = 0, w = 0;
            if (!succ(s, i, to, w))
              break;
            if (to != DEAD && depth[to] + w > depth[s])
            {
              depth[s] = depth[to] + w;
              changed = true;
            }
          }
      }
      out.max_match_len = depth[0];
    }
  }
  return UGX_OK;
}

// ---- line-resetting search automaton (`-c`) --------------------------------------------------------------

void build_search_dfa(const HostDfa& dfa, SearchDfa& out, uint32_t max_bytes)
{
  out = SearchDfa();
  if (dfa.has_meta)
  {
    out.refusal = UGX_SEARCH_META;
    return;
  }
  if (dfa.nstates == 0 || dfa.accept[0] != 0)
  {
    out.refusal = UGX_SEARCH_ACC0;
    return;
  }
  const uint32_t ncls = dfa.ncls;
  // one anchored transition as attempt_table (stream_count.cu) takes it: -1 the attempt fails, -2 it matches, else the
  // attempt is still undecided in the returned state
  auto outcome = [&](uint32_t s, uint32_t c) -> int32_t {
    const uint32_t t = dfa.next[static_cast<size_t>(s) * ncls + c];
    if (t >= dfa.first_acc)
    {
      if (t == DEAD)
        return -1;
      if (t < dfa.first_leaf)
        return -2;
      return (dfa.accept[t] & 0x7fffffffu) != 0 ? -2 : -1; // a leaf: a match unless it is a dead end
    }
    return static_cast<int32_t>(t);
  };

  // decision depth: the undecided states reachable from the start state must form an acyclic graph; D = its longest path
  // (in edges) plus one, so an attempt has decided after at most D bytes
  std::vector<uint8_t> color(dfa.nstates, 0); // 0 unseen, 1 on the DFS stack, 2 done
  std::vector<uint32_t> longest(dfa.nstates, 0);
  std::vector<std::pair<uint32_t, uint32_t>> stack{{0u, 0u}};
  color[0] = 1;
  while (!stack.empty())
  {
    auto& top = stack.back();
    if (top.second < ncls)
    {
      const int32_t o = outcome(top.first, top.second++);
      if (o < 0)
        continue;
      if (color[o] == 1)
      {
        out.refusal = UGX_SEARCH_CYCLE;
        return;
      }
      if (color[o] == 0)
      {
        color[o] = 1;
        stack.push_back({static_cast<uint32_t>(o), 0u});
      }
      continue;
    }
    const uint32_t s = top.first;
    uint32_t lp = 0;
    for (uint32_t c = 0; c < ncls; ++c)
    {
      const int32_t o = outcome(s, c);
      if (o >= 0 && longest[o] + 1 > lp)
        lp = longest[o] + 1;
    }
    longest[s] = lp;
    color[s] = 2;
    stack.pop_back();
  }
  out.depth = longest[0] + 1;
  if (out.depth > SEARCH_MAX_DEPTH)
  {
    out.refusal = UGX_SEARCH_DEPTH;
    return;
  }
  // '\n' must end every undecided attempt without a match (check_scope already rejects live '\n' edges), so that the
  // reset on '\n' is what the attempts themselves do
  const uint32_t nlc = dfa.cls[static_cast<uint8_t>('\n')];
  for (uint32_t s = 0; s < dfa.nstates; ++s)
    if (color[s] == 2 && outcome(s, nlc) != -1)
    {
      out.refusal = UGX_SEARCH_NEWLINE;
      return;
    }

  // classes: the anchored ones, '\n' split off when it shares its class (MATCHED resets on '\n' only)
  bool shared = false;
  for (uint32_t b = 0; b < 256; ++b)
    shared = shared || (b != '\n' && dfa.cls[b] == nlc);
  const uint32_t nc = shared ? ncls + 1 : ncls;
  if (nc > 256)
  {
    out.refusal = UGX_SEARCH_SIZE; // the class map holds bytes
    return;
  }
  const uint32_t nl_class = shared ? ncls : nlc;
  memcpy(out.cls, dfa.cls, 256);
  out.cls[static_cast<uint8_t>('\n')] = static_cast<uint8_t>(nl_class);

  // subset construction: state 0 = MATCHED, state 1 = the empty set
  const uint32_t max_raw = 1u << 18;
  std::map<std::vector<uint16_t>, uint32_t> id_of;
  std::vector<std::vector<uint16_t>> sets{{}, {}};
  std::vector<uint32_t> raw; // [raw states * nc]
  id_of[{}] = 1;
  std::vector<uint16_t> nxt;
  for (uint32_t s = 0; s < sets.size(); ++s)
  {
    raw.resize(static_cast<size_t>(sets.size()) * nc, 0);
    for (uint32_t c = 0; c < nc; ++c)
    {
      uint32_t to;
      if (c == nl_class)
        to = 1;
      else if (s == 0)
        to = 0;
      else
      {
        const uint32_t ac = c == ncls ? nlc : c;
        bool matched = false;
        nxt.clear();
        const int32_t o0 = outcome(0, ac); // the attempt that starts at this byte
        matched = o0 == -2;
        if (o0 >= 0)
          nxt.push_back(static_cast<uint16_t>(o0));
        for (uint16_t e : sets[s])
        {
          const int32_t o = outcome(e, ac);
          matched = matched || o == -2;
          if (o >= 0)
            nxt.push_back(static_cast<uint16_t>(o));
        }
        if (matched)
          to = 0;
        else
        {
          std::sort(nxt.begin(), nxt.end());
          nxt.erase(std::unique(nxt.begin(), nxt.end()), nxt.end());
          auto it = id_of.find(nxt);
          if (it != id_of.end())
            to = it->second;
          else
          {
            if (sets.size() >= max_raw)
            {
              out.refusal = UGX_SEARCH_SIZE;
              return;
            }
            to = static_cast<uint32_t>(sets.size());
            id_of.emplace(nxt, to);
            sets.push_back(nxt);
            raw.resize(static_cast<size_t>(sets.size()) * nc, 0);
          }
        }
      }
      raw[static_cast<size_t>(s) * nc + c] = to;
    }
  }
  const uint32_t nraw = static_cast<uint32_t>(sets.size());

  // Moore minimisation; MATCHED is alone in its block from the start
  std::vector<uint32_t> block(nraw), nblock(nraw);
  for (uint32_t s = 0; s < nraw; ++s)
    block[s] = s == 0 ? 0u : 1u;
  uint32_t nblocks = nraw > 1 ? 2 : 1;
  for (;;)
  {
    std::map<std::vector<uint32_t>, uint32_t> sig_id;
    std::vector<uint32_t> sig(nc + 1);
    // numbered in state order: MATCHED and the empty set keep blocks 0 and 1
    auto visit = [&](uint32_t s) {
      sig[0] = block[s];
      for (uint32_t c = 0; c < nc; ++c)
        sig[c + 1] = block[raw[static_cast<size_t>(s) * nc + c]];
      auto it = sig_id.find(sig);
      if (it == sig_id.end())
        it = sig_id.emplace(sig, static_cast<uint32_t>(sig_id.size())).first;
      nblock[s] = it->second;
    };
    for (uint32_t s = 0; s < nraw; ++s)
      visit(s);
    const uint32_t nb = static_cast<uint32_t>(sig_id.size());
    block.swap(nblock);
    if (nb == nblocks)
      break;
    nblocks = nb;
  }
  out.nstates = nblocks;
  out.ncls = nc;
  if (static_cast<uint64_t>(nblocks) * nc > 65536u || out.table_bytes() > max_bytes)
  {
    out.refusal = UGX_SEARCH_SIZE;
    return;
  }
  out.next.assign(static_cast<size_t>(nblocks) * nc, 0);
  for (uint32_t s = 0; s < nraw; ++s)
    for (uint32_t c = 0; c < nc; ++c)
      out.next[static_cast<size_t>(block[s]) * nc + c] = static_cast<uint16_t>(block[raw[static_cast<size_t>(s) * nc + c]] * nc);
}

// ---- k-gram viability ----------------------------------------------------------------------------------

void build_viability(const HostDfa& dfa, Viability& v, uint32_t max_bits)
{
  v = Viability();
  if (dfa.has_meta || dfa.nstates == 0 || dfa.accept[0] != 0)
    return;
  const uint32_t ncls = dfa.ncls;
  auto step = [&](uint32_t s, uint32_t b) -> uint16_t { return dfa.next[static_cast<size_t>(s) * ncls + dfa.cls[b]]; };
  // ids of a level: bytes that every state of `level` treats alike share an id; false when there are too many
  auto assign_ids = [&](const std::vector<uint32_t>& level, uint32_t (&ids)[256], std::vector<uint8_t>& reps) -> bool {
    std::map<std::vector<uint16_t>, uint32_t> id_of;
    reps.clear();
    for (uint32_t b = 0; b < 256; ++b)
    {
      std::vector<uint16_t> col(level.size());
      for (size_t j = 0; j < level.size(); ++j)
        col[j] = step(level[j], b);
      auto it = id_of.find(col);
      if (it == id_of.end())
      {
        it = id_of.emplace(col, static_cast<uint32_t>(reps.size())).first;
        reps.push_back(static_cast<uint8_t>(b));
      }
      ids[b] = it->second;
    }
    return reps.size() <= 255;
  };
  auto targets = [&](const std::vector<uint32_t>& level) {
    std::vector<uint8_t> seen(dfa.nstates, 0);
    std::vector<uint32_t> out;
    for (uint32_t s : level)
      for (uint32_t c = 0; c < ncls; ++c)
      {
        const uint16_t t = dfa.next[static_cast<size_t>(s) * ncls + c];
        if (t != DEAD && !seen[t])
        {
          seen[t] = 1;
          out.push_back(t);
        }
      }
    return out;
  };
  // ---- bytes one and two: the pair table of state codes
  uint32_t id0[256], id1[256], id2[256] = {0}, id3[256] = {0};
  std::vector<uint8_t> rep0, rep1, rep2, rep3;
  const std::vector<uint32_t> l0{0u};
  if (!assign_ids(l0, id0, rep0))
    return;
  const std::vector<uint32_t> l1 = targets(l0);
  if (l1.empty() || !assign_ids(l1, id1, rep1) || rep0.size() * rep1.size() > 16384)
    return;
  const uint32_t n0 = static_cast<uint32_t>(rep0.size()), n1 = static_cast<uint32_t>(rep1.size());
  std::vector<uint32_t> s2; // distinct live, not yet accepting states after two bytes
  std::map<uint32_t, uint32_t> s2_id;
  std::vector<int> raw(static_cast<size_t>(n0) * n1, 0); // 0 dead, -1 accepted, 1 + index into s2
  for (uint32_t a = 0; a < n0; ++a)
    for (uint32_t b = 0; b < n1; ++b)
    {
      int code = 0;
      const uint16_t t1 = step(0, rep0[a]);
      if (t1 != DEAD)
      {
        if (dfa.accept[t1] != 0)
          code = -1;
        else
        {
          const uint16_t t2 = step(t1, rep1[b]);
          if (t2 != DEAD)
          {
            if (dfa.accept[t2] != 0)
              code = -1;
            else
            {
              auto it = s2_id.find(t2);
              if (it == s2_id.end())
              {
                it = s2_id.emplace(t2, static_cast<uint32_t>(s2.size())).first;
                s2.push_back(t2);
              }
              code = static_cast<int>(it->second) + 1;
            }
          }
        }
      }
      raw[static_cast<size_t>(a) * n1 + b] = code;
    }
  if (s2.size() > 253)
  {
    // too many states after two bytes for one byte of code: every live pair just stays viable
    for (auto& c : raw)
      c = c != 0 ? -1 : 0;
    s2.clear();
  }
  v.k = 2;
  // ---- bytes three and four: a bit table over (state code, id2, id3)
  uint32_t n2 = 1, n3 = 1;
  if (!s2.empty() && assign_ids(s2, id2, rep2) && static_cast<uint64_t>(s2.size() + 2) * rep2.size() <= max_bits)
  {
    v.k = 3;
    n2 = static_cast<uint32_t>(rep2.size());
    const std::vector<uint32_t> l3 = targets(s2);
    if (!l3.empty() && assign_ids(l3, id3, rep3) && static_cast<uint64_t>(s2.size() + 2) * n2 * rep3.size() <= max_bits &&
        static_cast<uint64_t>(n2) * rep3.size() <= 0xffff)
    {
      v.k = 4;
      n3 = static_cast<uint32_t>(rep3.size());
    }
    else
      memset(id3, 0, sizeof(id3));
  }
  else
    memset(id2, 0, sizeof(id2));
  const uint32_t accepted = static_cast<uint32_t>(s2.size()) + 1;
  v.stride = n2 * n3;
  v.pair.assign(raw.size(), 0);
  for (size_t i = 0; i < raw.size(); ++i)
    v.pair[i] = static_cast<uint8_t>(raw[i] < 0 ? accepted : raw[i]);
  for (uint32_t b = 0; b < 256; ++b)
  {
    v.t01[b] = (id0[b] * n1) | (id1[b] << 16);
    v.t23[b] = (v.k >= 3 ? id2[b] * n3 : 0u) | ((v.k >= 4 ? id3[b] : 0u) << 16);
  }
  const uint64_t total = static_cast<uint64_t>(accepted + 1) * v.stride;
  v.bits.assign((total + 31) / 32, 0);
  auto set_bit = [&](uint64_t idx) { v.bits[idx >> 5] |= 1u << (idx & 31); };
  for (uint32_t code = 1; code <= accepted; ++code)
    for (uint32_t c2 = 0; c2 < n2; ++c2)
      for (uint32_t c3 = 0; c3 < n3; ++c3)
      {
        bool ok = true;
        if (code != accepted && v.k >= 3)
        {
          const uint16_t t3 = step(s2[code - 1], rep2[c2]);
          if (t3 == DEAD)
            ok = false;
          else if (dfa.accept[t3] == 0 && v.k >= 4)
            ok = step(t3, rep3[c3]) != DEAD;
        }
        if (ok)
          set_bit((static_cast<uint64_t>(code) * n2 + c2) * n3 + c3);
      }
}

// ---- first-stage filter planning -------------------------------------------------------------------

namespace {

// a rough prior of byte frequencies in text (per mille), used only to rank filter choices
double byte_prior(uint32_t c)
{
  static const double lower[26] = {65, 12, 22, 34, 102, 18, 16, 49, 56, 1, 6, 32, 19, 54, 60, 15, 1, 48, 51, 73, 22, 8, 19, 1, 16, 1};
  if (c >= 'a' && c <= 'z')
    return lower[c - 'a'];
  if (c >= 'A' && c <= 'Z')
    return lower[c - 'A'] * 0.05 + 0.5;
  if (c == ' ')
    return 150;
  if (c >= '0' && c <= '9')
    return 8;
  if (c == '\n')
    return 20;
  if (c >= 0x80)
    return 1.5;
  if (c < 0x20 || c == 0x7f)
    return 0.2;
  return 3;
}

uint32_t to_ppm(double x)
{
  if (x < 0)
    x = 0;
  if (x > 1)
    x = 1;
  return static_cast<uint32_t>(x * 1e6);
}

// necessary condition on the FIRST byte of a window for Pattern::predict_match to pass
// (include/reflex/pattern.h:366-401): PMH step 0 reads bit 0 of pmh[c0]; PM4 passes iff, with p7..p0 the gathered
// bits,  !p7 | (!p6 & (!p5 | ...)) | ...  — c0 can start a passing window only if !p7, or !p6, or some second byte
// gives !p5.
bool can_start(const ugx_prefilter& pf, uint32_t c0)
{
  if (pf.min >= 4)
    return (pf.pmh[c0] & 1u) == 0;
  const uint8_t* pred = pf.pma;
  if ((pred[c0] & 0xc0) != 0xc0)
    return true;
  for (uint32_t c1 = 0; c1 < 256; ++c1)
    if ((pred[((c0 << 3) ^ c1) & (UGX_HASH - 1)] & 0x20) == 0)
      return true;
  return false;
}

// add a term: `in_set[c]` says whether byte c passes; returns the prior pass rate of the set
double add_term(FilterPlan& plan, uint32_t off, const bool (&in_set)[256])
{
  const uint32_t t = plan.nterms++;
  plan.t_off[t] = off;
  double pass = 0;
  for (uint32_t c = 0; c < 256; ++c)
  {
    if (in_set[c])
      pass += byte_prior(c) / 1000.0;
    else
      plan.lut[c] |= 1u << (8 * t);
  }
  return pass > 1.0 ? 1.0 : pass;
}

} // namespace

bool prefilter_never_fires(const ugx_prefilter& pf, int adv)
{
  if (adv != UGX_ADV_MIN1 && adv != UGX_ADV_MIN2 && adv != UGX_ADV_MIN3 && adv != UGX_ADV_MIN4)
    return false;
  // every one of these routines requires bit j of tap[pair(k + j)] to be clear for all j < depth (MIN1: j = 0)
  const uint32_t depth = pf.min < 1 ? 1 : pf.min;
  for (uint32_t j = 0; j < depth && j < 8; ++j)
  {
    bool some = false;
    for (uint32_t i = 0; i < UGX_BTAP && !some; ++i)
      some = ((pf.tap[i] >> j) & 1u) == 0;
    if (!some)
      return true;
  }
  return false;
}

// ---- does the prefilter accept every position at which a non-empty match starts? -------------------------------------
// The candidate predicates of device_pattern.cuh, restated on the host in their interior form (far enough from the end of
// the buffer that no end-of-buffer clause applies), read a fixed number E of bytes at the position.  Every match start
// is either an E-byte DFA path that is still alive or a shorter accepted prefix followed by anything; enumerating those
// strings and evaluating the predicate on each PROVES {p : D(p) > 0} is a subset of the candidates (or finds a
// counter-example: config 3's false negatives).  The count-lines kernels may then skip the predicate: a line has a match
// iff some position of it starts one.  Bounded: more than `cap` strings = not proven.
namespace {

struct CoverCheck {
  const HostDfa& dfa;
  const ugx_prefilter& pf;
  int adv;
  uint32_t extent;
  uint64_t budget;
  const uint8_t* pred;
  uint32_t pin_a[8] = {0}, pin_b[8] = {0};
  uint8_t s[320];
  bool ok = true;

  static uint32_t hash3(uint32_t h, uint32_t b) { return ((h << 3) ^ b) & (UGX_HASH - 1); }
  static bool in(const uint32_t* set, uint32_t c) { return (set[c >> 5] >> (c & 31)) & 1u; }
  bool pm4(const uint8_t* p) const
  {
    const uint32_t h1 = hash3(p[0], p[1]), h2 = hash3(h1, p[2]), h3 = hash3(h2, p[3]);
    const uint32_t q = (pred[p[0]] & 0xc0u) | (pred[h1] & 0x30u) | (pred[h2] & 0x0cu) | (pred[h3] & 0x03u);
    const uint32_t r = ((((((q >> 2) | q) >> 2) | q) >> 1) | q) & 0xffu;
    return r != 0xffu;
  }
  bool pmh(const uint8_t* p, uint32_t n) const
  {
    uint32_t h = p[0];
    uint32_t f = pred[h] & 1u, bit = 2;
    for (uint32_t j = 1; j < n; ++j, bit <<= 1)
    {
      h = hash3(h, p[j]);
      f |= pred[h] & bit;
    }
    return f == 0;
  }
  bool tapbit(const uint8_t* p, uint32_t j) const { return (pf.tap[(p[0] ^ (static_cast<uint32_t>(p[1]) << 6)) & (UGX_BTAP - 1)] >> j) & 1u; }
  bool literal() const { return memcmp(s, pf.chr, pf.len) == 0; }

  bool cand() const
  {
    const uint32_t min = pf.min, len = pf.len, lcp = pf.lcp, lcs = pf.lcs;
    switch (adv)
    {
      case UGX_ADV_PIN1_ONE: return s[0] == pf.chr[0] && pm4(s);
      case UGX_ADV_PIN1_PMA: return s[lcp] == pf.chr[0] && s[lcs] == pf.chr[1] && pm4(s);
      case UGX_ADV_PIN1_PMH: return s[lcp] == pf.chr[0] && s[lcs] == pf.chr[1] && pmh(s, min);
      case UGX_ADV_PIN_ONE: return in(pin_a, s[0]) && pm4(s);
      case UGX_ADV_PIN_PMA: return in(pin_a, s[lcp]) && in(pin_b, s[lcs]) && pm4(s);
      case UGX_ADV_PIN_PMH: return in(pin_a, s[lcp]) && in(pin_b, s[lcs]) && pmh(s, min);
      case UGX_ADV_MIN1: return !tapbit(s, 0) && pm4(s);
      case UGX_ADV_MIN2: return !tapbit(s, 0) && !tapbit(s + 1, 1) && pm4(s);
      case UGX_ADV_MIN3: return !tapbit(s, 0) && !tapbit(s + 1, 1) && !tapbit(s + 2, 2) && pm4(s);
      case UGX_ADV_MIN4:
        for (uint32_t j = 0; j < min; ++j)
          if (tapbit(s + j, j))
            return false;
        return pmh(s, min);
      case UGX_ADV_PMA: return pm4(s);
      case UGX_ADV_CHAR: return s[0] == pf.chr[0];
      case UGX_ADV_CHAR_PMA: return s[0] == pf.chr[0] && pm4(s + 1);
      case UGX_ADV_CHAR_PMH: return s[0] == pf.chr[0] && pmh(s + 1, min);
      case UGX_ADV_STRING: return literal();
      case UGX_ADV_STRING_PMA: return literal() && pm4(s + len);
      case UGX_ADV_STRING_PMH: return literal() && pmh(s + len, min);
      case UGX_ADV_NONE: return true;
      default: return false;
    }
  }

  void leaf()
  {
    if (budget == 0)
    {
      ok = false;
      return;
    }
    --budget;
    if (!cand())
      ok = false;
  }

  // PM4 on a window whose first L bytes (1 <= L <= 3) are p[0..L) and whose other bytes are ANYTHING: the verdict of
  // predict_match depends on the unknown bytes only through the two table bits of each unknown level, so "passes for
  // all 4^(4-L) values of those bits" is a sufficient condition for "passes whatever follows"
  bool pm4_whatever_follows(const uint8_t* p, uint32_t L) const
  {
    uint32_t q = pred[p[0]] & 0xc0u;
    uint32_t h = p[0];
    if (L >= 2)
    {
      h = hash3(h, p[1]);
      q |= pred[h] & 0x30u;
    }
    if (L >= 3)
    {
      h = hash3(h, p[2]);
      q |= pred[h] & 0x0cu;
    }
    const uint32_t free_bits = L == 1 ? 0x3fu : L == 2 ? 0x0fu : 0x03u;
    for (uint32_t v = 0; v <= free_bits; ++v)
    {
      const uint32_t qq = q | v;
      const uint32_t r = ((((((qq >> 2) | qq) >> 2) | qq) >> 1) | qq) & 0xffu;
      if (r == 0xffu)
        return false;
    }
    return true;
  }

  // the routines whose interior test is [needle bytes] && PM4 on the window at offset `win`: does s[0..depth) followed by
  // anything pass?  (sufficient, not necessary)
  bool passes_whatever_follows(uint32_t depth) const
  {
    uint32_t win = 0;
    switch (adv)
    {
      case UGX_ADV_PMA: break;
      case UGX_ADV_PIN_ONE:
        if (!in(pin_a, s[0]))
          return false;
        break;
      case UGX_ADV_PIN1_ONE:
        if (s[0] != pf.chr[0])
          return false;
        break;
      case UGX_ADV_PIN_PMA:
        if (pf.lcp >= depth || pf.lcs >= depth || !in(pin_a, s[pf.lcp]) || !in(pin_b, s[pf.lcs]))
          return false;
        break;
      case UGX_ADV_PIN1_PMA:
        if (pf.lcp >= depth || pf.lcs >= depth || s[pf.lcp] != pf.chr[0] || s[pf.lcs] != pf.chr[1])
          return false;
        break;
      case UGX_ADV_CHAR_PMA:
        if (s[0] != pf.chr[0])
          return false;
        win = 1;
        break;
      case UGX_ADV_STRING_PMA:
        if (depth < pf.len || !literal())
          return false;
        win = pf.len;
        break;
      case UGX_ADV_MIN1:
      case UGX_ADV_MIN2:
      case UGX_ADV_MIN3:
      {
        // bitap step j reads the byte pair (j, j + 1): known bytes as they are, the first unknown byte as all 256 values
        const uint32_t steps = adv == UGX_ADV_MIN1 ? 1 : adv == UGX_ADV_MIN2 ? 2 : 3;
        for (uint32_t j = 0; j < steps; ++j)
        {
          if (j >= depth)
            return false;
          if (j + 1 < depth)
          {
            if (tapbit(s + j, j))
              return false;
          }
          else
            for (uint32_t b = 0; b < 256; ++b)
              if ((pf.tap[(s[j] ^ (b << 6)) & (UGX_BTAP - 1)] >> j) & 1u)
                return false;
        }
        break;
      }
      default: return false;
    }
    if (depth <= win || depth >= win + 4)
      return false;
    return pm4_whatever_follows(s + win, depth - win);
  }

  // every completion of s[0..depth) to `extent` bytes
  void pad(uint32_t depth)
  {
    if (depth == extent)
      return leaf();
    if (passes_whatever_follows(depth))
    {
      if (budget == 0)
        ok = false;
      else
        --budget;
      return;
    }
    if (extent - depth > 2)
    {
      ok = false; // 2^24 completions and more: not enumerated
      return;
    }
    for (uint32_t b = 0; b < 256 && ok; ++b)
    {
      s[depth] = static_cast<uint8_t>(b);
      pad(depth + 1);
    }
  }

  void walk(uint32_t state, uint32_t depth)
  {
    if (!ok)
      return;
    if (depth > 0 && dfa.accept[state] != 0)
      return pad(depth); // a match ends here: whatever follows, the position starts a match
    if (depth == extent)
      return leaf();
    if (budget == 0)
    {
      ok = false;
      return;
    }
    --budget;
    for (uint32_t b = 0; b < 256 && ok; ++b)
    {
      const uint16_t nx = dfa.next[static_cast<size_t>(state) * dfa.ncls + dfa.cls[b]];
      if (nx == DEAD)
        continue;
      s[depth] = static_cast<uint8_t>(b);
      walk(nx, depth + 1);
    }
  }
};

} // namespace

bool prefilter_covers_matches(const HostDfa& dfa, const ugx_prefilter& pf, int adv, uint32_t matcher_flags, uint32_t cap)
{
  if (dfa.has_meta || pf.one || (matcher_flags & UGX_OPT_W) != 0)
    return false; // META edges and option W make D(p) depend on more than the bytes at p; `one`: the predicate IS the match
  // (look-back only ADDS positions to the attempt set, A = cand | (cbk & A + 1): cand covering the match starts is enough)
  const uint32_t min = pf.min, len = pf.len;
  uint32_t e;
  switch (adv)
  {
    case UGX_ADV_PIN1_ONE: case UGX_ADV_PIN_ONE: case UGX_ADV_PMA:
    case UGX_ADV_MIN1: case UGX_ADV_MIN2: case UGX_ADV_MIN3: e = 4; break;
    case UGX_ADV_PIN1_PMA: case UGX_ADV_PIN_PMA: e = 4; break;
    case UGX_ADV_PIN1_PMH: case UGX_ADV_PIN_PMH: e = min; break;
    case UGX_ADV_MIN4: e = min + 1; break;
    case UGX_ADV_CHAR: e = 1; break;
    case UGX_ADV_CHAR_PMA: e = 5; break;
    case UGX_ADV_CHAR_PMH: e = 1 + min; break;
    case UGX_ADV_STRING: e = len; break;
    case UGX_ADV_STRING_PMA: e = len + 4; break;
    case UGX_ADV_STRING_PMH: e = len + min; break;
    case UGX_ADV_NONE: return true;
    default: return false;
  }
  if (adv == UGX_ADV_PIN1_PMA || adv == UGX_ADV_PIN_PMA || adv == UGX_ADV_PIN1_PMH || adv == UGX_ADV_PIN_PMH)
  {
    if (pf.lcp + 1 > e)
      e = pf.lcp + 1;
    if (pf.lcs + 1 > e)
      e = pf.lcs + 1;
  }
  if (e == 0 || e > 24) // the kernels guarantee 24 readable bytes after an interior position
    return false;
  CoverCheck c{dfa, pf, adv, e, cap, pf.min < 4 ? pf.pma : pf.pmh};
  if (pf.len == 0 && pf.pin >= 1 && pf.pin <= 16)
    for (uint32_t i = 0; i < pf.pin; ++i)
    {
      const uint32_t a = pf.chr[i], b = pf.chr[pf.pin + i];
      c.pin_a[a >> 5] |= 1u << (a & 31);
      c.pin_b[b >> 5] |= 1u << (b & 31);
    }
  memset(c.s, 0, sizeof(c.s));
  c.walk(0, 0);
  return c.ok;
}

void plan_filter(const ugx_prefilter& pf, int adv, FilterPlan& plan)
{
  memset(&plan, 0, sizeof(plan));
  plan.kind = FK_ALL;
  plan.est_pass_ppm = 1000000;
  // hashed-predictor terms: steps j >= 3 of predict_match read pmh[g(k + j)] with g a hash of 4 text bytes only
  if (pf.min >= 4 && (adv == UGX_ADV_PIN1_PMH || adv == UGX_ADV_PIN_PMH || adv == UGX_ADV_MIN4 || adv == UGX_ADV_CHAR_PMH))
  {
    plan.h4_terms = pf.min - 3 > 3 ? 3 : pf.min - 3;
    plan.h4_shift = adv == UGX_ADV_CHAR_PMH ? 1 : 0;
  }
  // PM4 two-byte term for the routines that call predict_match PM4 on every interior candidate and have no
  // selective byte-set term of their own
  if (pf.min < 4 && (adv == UGX_ADV_PMA || adv == UGX_ADV_MIN1 || adv == UGX_ADV_MIN2 || adv == UGX_ADV_MIN3))
  {
    plan.pm2 = 1;
    plan.pm2_shift = 0;
  }
  switch (adv)
  {
    case UGX_ADV_STRING:
    case UGX_ADV_STRING_PMA:
    case UGX_ADV_STRING_PMH:
    {
      // anchor 0 is the first byte (compared without a shift).  Anchor 1 comes from bytes 1..12 (the register
      // window holds 12 halo bytes): the farthest word-aligned offset (12, 8, 4: no funnel shift, and far from
      // anchor 0, so less correlated with it) whose pair is selective enough under the byte prior, else the
      // rarest byte (ties: the farthest).
      const uint32_t span = pf.len < 13 ? pf.len : 13;
      uint32_t best[2] = {0, 0};
      double score[2] = {byte_prior(pf.chr[0]), 1e9};
      for (uint32_t i = 1; i < span; ++i)
      {
        const double f = byte_prior(pf.chr[i]);
        if (f <= score[1])
        {
          score[1] = f;
          best[1] = i;
        }
      }
      if (span == 1)
        score[1] = 1000.0;
      for (uint32_t i = 12; i >= 4; i -= 4)
      {
        if (i >= span)
          continue;
        const double f = byte_prior(pf.chr[i]);
        if (score[0] * f / 1e6 <= 2e-4 || f <= 1.5 * score[1])
        {
          score[1] = f;
          best[1] = i;
          break;
        }
      }
      if (!pf.one || adv != UGX_ADV_STRING)
      {
        // literal prefix followed by more pattern: the same two bytes as byte-set terms
        plan.kind = FK_LUT;
        bool s0[256] = {false}, s1[256] = {false};
        s0[pf.chr[0]] = true;
        double est = add_term(plan, 0, s0);
        if (span > 1)
        {
          uint32_t j = best[1] <= 8 ? best[1] : 1;
          s1[pf.chr[j]] = true;
          est *= add_term(plan, j, s1);
        }
        plan.est_pass_ppm = to_ppm(est);
        return;
      }
      plan.kind = FK_ANCHOR2;
      for (int a = 0; a < 2; ++a)
      {
        plan.a_off[a] = best[a];
        plan.a_chr[a] = pf.chr[best[a]] * 0x01010101u;
      }
      plan.est_pass_ppm = to_ppm(score[0] / 1000.0 * (span > 1 ? score[1] / 1000.0 : 1.0));
      return;
    }
    case UGX_ADV_CHAR:
    case UGX_ADV_CHAR_PMA:
    case UGX_ADV_CHAR_PMH:
    {
      plan.kind = FK_LUT;
      bool set0[256] = {false};
      set0[pf.chr[0]] = true;
      double est = add_term(plan, 0, set0);
      if (adv != UGX_ADV_CHAR)
      {
        bool set1[256];
        for (uint32_t c = 0; c < 256; ++c)
          set1[c] = can_start(pf, c); // the predictor looks at k + 1
        est *= add_term(plan, 1, set1);
      }
      plan.est_pass_ppm = to_ppm(est);
      return;
    }
    case UGX_ADV_PIN1_ONE:
    case UGX_ADV_PIN_ONE:
    {
      // needle set at k, and the predictor's first-byte condition at the same byte
      plan.kind = FK_LUT;
      bool set0[256] = {false};
      for (uint32_t i = 0; i < pf.pin; ++i)
        set0[pf.chr[i]] = true;
      for (uint32_t c = 0; c < 256; ++c)
        set0[c] = set0[c] && can_start(pf, c);
      plan.est_pass_ppm = to_ppm(add_term(plan, 0, set0));
      return;
    }
    case UGX_ADV_PIN1_PMA:
    case UGX_ADV_PIN1_PMH:
    case UGX_ADV_PIN_PMA:
    case UGX_ADV_PIN_PMH:
    {
      // needle sets at k + lcp and k + lcs, and the predictor's first-byte condition at k
      plan.kind = FK_LUT;
      bool seta[256] = {false}, setb[256] = {false}, setz[256];
      for (uint32_t i = 0; i < pf.pin; ++i)
      {
        seta[pf.chr[i]] = true;
        setb[pf.chr[pf.pin + i]] = true;
      }
      for (uint32_t c = 0; c < 256; ++c)
        setz[c] = can_start(pf, c);
      double est = 1.0;
      if (pf.lcp == 0)
        for (uint32_t c = 0; c < 256; ++c)
          seta[c] = seta[c] && setz[c];
      else if (pf.lcs == 0)
        for (uint32_t c = 0; c < 256; ++c)
          setb[c] = setb[c] && setz[c];
      est *= add_term(plan, pf.lcp, seta);
      if (pf.lcs != pf.lcp)
        est *= add_term(plan, pf.lcs, setb);
      if (pf.lcp != 0 && pf.lcs != 0)
        est *= add_term(plan, 0, setz);
      plan.est_pass_ppm = to_ppm(est);
      return;
    }
    case UGX_ADV_MIN1:
    case UGX_ADV_MIN2:
    case UGX_ADV_MIN3:
    case UGX_ADV_MIN4:
    {
      // bitap over hashed byte pairs: step j reads bit j of tap[pair(k + j)].  Byte-level necessary condition:
      // byte (k + j) must be the first byte of SOME pair that passes step j.
      const uint32_t depth = pf.min < 1 ? 1 : pf.min;
      plan.kind = FK_LUT;
      double est = 1.0;
      for (uint32_t j = 0; j < depth && plan.nterms < FILTER_MAX_TERMS; ++j)
      {
        bool setj[256];
        for (uint32_t c = 0; c < 256; ++c)
        {
          setj[c] = false;
          for (uint32_t d = 0; d < 256 && !setj[c]; ++d)
            setj[c] = ((pf.tap[(c ^ (d << 6)) & (UGX_BTAP - 1)] >> j) & 1u) == 0;
        }
        est *= add_term(plan, j, setj);
      }
      plan.est_pass_ppm = to_ppm(est);
      return;
    }
    case UGX_ADV_PMA:
    {
      plan.kind = FK_LUT;
      bool set0[256];
      for (uint32_t c = 0; c < 256; ++c)
        set0[c] = can_start(pf, c);
      plan.est_pass_ppm = to_ppm(add_term(plan, 0, set0));
      return;
    }
    default:
      return;
  }
}

int check_scope(const HostDfa& dfa, const ugx_prefilter& pf, uint32_t matcher_flags, std::string& err)
{
  if (dfa.newline_live)
  {
    err = "the DFA has a transition on '\\n': matches are not line-local";
    return UGX_E_UNSUPPORTED;
  }
  if (pf.lbk != 0 && (pf.cbk['\n' >> 3] >> ('\n' & 7) & 1))
  {
    err = "look-back set contains '\\n'";
    return UGX_E_UNSUPPORTED;
  }
  if (pf.len > 255 || pf.min > 8 || pf.pin > 16 || (pf.len == 0 && pf.pin > 0 && (pf.lcp >= 8 || pf.lcs >= 8)))
  {
    err = "prefilter fields out of range";
    return UGX_E_INVALID;
  }
  if (pf.len > 0)
    for (uint32_t i = 0; i < pf.len; ++i)
      if (pf.chr[i] == '\n')
      {
        err = "literal prefix contains '\\n'";
        return UGX_E_UNSUPPORTED;
      }
  return UGX_OK;
}

} // namespace ugx
