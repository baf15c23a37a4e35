// pattern_host.hpp — host-side "DFA export": reflex::Pattern opcode words -> dense,
// byte-class-compressed transition table + the prefilter routine selection.
// No CUDA here: this part is unit-tested on the CPU.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include "../../include/ugrep_b200.h"
#include "filter_plan.hpp"

namespace ugx {

constexpr uint32_t OP_HALT = 0x00FFFFFFu;
constexpr uint32_t IDX_HALT = 0xFFFFu;
constexpr uint32_t IDX_LONG = 0xFFFEu;
constexpr uint16_t DEAD = 0xFFFFu;

// opcode codec, /root/reference/include/reflex/pattern.h:1155-1247
inline bool op_is_goto(uint32_t op) { return (op << 8) >= (op & 0xff000000u); }

struct MetaEdge {
  uint32_t code;   // META code - 0x100 (pattern.h:930-952)
  uint32_t target; // dense state id
};

struct HostDfa {
  uint32_t nstates = 0;
  uint32_t ncls = 0;
  uint8_t cls[256] = {0};          // byte -> equivalence class
  std::vector<uint16_t> next;      // [nstates * ncls], DEAD = no transition
  std::vector<uint32_t> accept;    // [nstates] accept index (TAKE), 0 = none
  std::vector<uint32_t> word_of;   // [nstates] opcode word index of the state
  std::vector<uint32_t> meta_off;  // [nstates + 1] offsets into metas
  std::vector<MetaEdge> metas;
  bool has_meta = false;
  bool newline_live = false;       // some state has a transition on '\n'
  bool to_start = false;           // some transition targets state 0 (start-loop skip, lib/matcher.cpp:504-527)
  // states are numbered: 0 = start, then non-accepting states with byte edges, then accepting states with
  // byte edges, then states without byte edges ("leaves": the interpreter halts there before reading)
  uint32_t first_acc = 0;          // ids >= first_acc (other than 0) are accepting or leaves
  uint32_t first_leaf = 0;         // ids >= first_leaf (other than 0) are leaves
  uint32_t max_match_len = 0;      // longest match in bytes; UINT32_MAX when the DFA has a cycle (unbounded)
  uint32_t table_bytes() const { return nstates * ncls * 2; }
};

// k-gram viability of an anchored attempt (span_scan.cu, stream_count.cu): position p can only start a match if the DFA,
// fed the k bytes at p, accepts on the way or is still alive after them.  Bytes are mapped to small per-level ids (two
// bytes get the same id at level i when every state reachable after i bytes treats them alike); the tables hold the ids
// pre-multiplied so that the device does two adds and two lookups per position:
//   code = pair[(t01[b0] & 0xffff) + (t01[b1] >> 16)]      0 = dead within two bytes, 1 + s = the s-th distinct state
//                                                         reached, `accepted` = accepted within two bytes (a row of ones)
//   viable = bit (code * stride + (t23[b2] & 0xffff) + (t23[b3] >> 16)) of `bits`
// k = 0: no table (META edges, accepting start state, too many ids).  A property of the DFA alone: it never changes which
// positions match, it only spares attempts that cannot.
struct Viability {
  uint32_t k = 0;               // bytes looked at: 0 (none), 2, 3 or 4
  uint32_t stride = 1;          // bits per state code: ids at level 2 times ids at level 3
  uint32_t t01[256] = {0};      // (id0 * n1) | id1 << 16
  uint32_t t23[256] = {0};      // (id2 * n3) | id3 << 16
  std::vector<uint8_t> pair;    // [n0 * n1] state codes
  std::vector<uint32_t> bits;   // [(states + 2) * stride] bits
};
void build_viability(const HostDfa& dfa, Viability& v, uint32_t max_bits = 1u << 18);

// Line-resetting search automaton for `-c` (stream_search.cu, DESIGN.md §4.3a).  A state is the set of anchored states of
// the attempts started earlier in the line that are still undecided, or MATCHED once one of them has decided "match" the
// way attempt_table decides it.  On each byte: add the start state, step every element; '\n' resets to the empty set.
// A line counts iff the automaton is MATCHED somewhere in it.  Minimised; `next` holds pre-multiplied row offsets
// (state * ncls) with MATCHED at offset 0 and the empty set at offset ncls, so the device steps by one add and one
// lookup and tests for success with `== 0`.
constexpr uint32_t SEARCH_MAX_DEPTH = 16;
constexpr uint32_t SEARCH_MAX_BYTES = 128 * 1024;

struct SearchDfa {
  uint32_t refusal = UGX_SEARCH_OK; // UGX_SEARCH_* (include/ugrep_b200.h)
  uint32_t depth = 0;          // D: the state at x depends only on bytes [x - (D - 1), x) of the line (MATCHED aside)
  uint32_t nstates = 0;        // minimised, MATCHED and the empty set included
  uint32_t ncls = 0;           // the anchored DFA's classes, plus one for '\n' when it shares its class
  uint8_t cls[256] = {0};
  std::vector<uint16_t> next;  // [nstates * ncls] pre-multiplied row offsets
  uint32_t table_bytes() const { return nstates * ncls * 2; }
};
// fills `out` (refusal = UGX_SEARCH_OK when the automaton applies; the route conditions are the caller's)
void build_search_dfa(const HostDfa& dfa, SearchDfa& out, uint32_t max_bytes = SEARCH_MAX_BYTES);

// Matcher::init_advance, /root/reference/lib/matcher.cpp:797-954
int select_advance(const ugx_prefilter& pf, uint32_t matcher_flags);

// returns UGX_OK or an error status; err receives a message
int flatten_dfa(const uint32_t* opc, uint32_t nop, HostDfa& out, std::string& err);

// true when the routine's tables admit no candidate position at all: a bitap step j < min_ that no byte pair passes
// (the advance_pattern_min* routines, lib/matcher.cpp:2235-2660, then never stop — config 3, SURVEY.md Q1)
bool prefilter_never_fires(const ugx_prefilter& pf, int adv);

// true when it is PROVEN (by enumeration over the DFA, bounded by `cap` strings) that every position at which a non-empty
// match starts passes the routine's candidate predicate, away from the end of the buffer
bool prefilter_covers_matches(const HostDfa& dfa, const ugx_prefilter& pf, int adv, uint32_t matcher_flags,
                              uint32_t cap = 1u << 18);

// first-stage filter of the position-parallel kernels (filter_plan.hpp)
void plan_filter(const ugx_prefilter& pf, int adv, FilterPlan& plan);

// checks that make the line-parallel scan exact for this pattern (DESIGN.md "line locality")
int check_scope(const HostDfa& dfa, const ugx_prefilter& pf, uint32_t matcher_flags, std::string& err);

} // namespace ugx
