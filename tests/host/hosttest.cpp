// TEST-ONLY library (never part of libgorpcuda.so, never shipped): interprets the tables that the product's
// definition compiler produces (CompactDfa + per-extraction TDFA) on the CPU, so that the host-side compile
// logic can be checked against the oracle without a GPU. The loops mirror kernels/kernels.cu (K2, K4).
#include <algorithm>
#include <cstdio>
#include <cstring>

#include "../../gorp_b200/csrc/host/fused.hpp"

using namespace gorp;

static int g_force_minimise = 0;
// 1: ht_run minimises every capture automaton (host/capture.hpp: minimise_tdfa) whatever path the definition takes
extern "C" void ht_set_force_minimise(int on) { g_force_minimise = on; }

extern "C" int ht_run(const void* blob, size_t len, const uint16_t* text, const int64_t* starts, const int64_t* ends, int64_t n,
                      int32_t* ext, int32_t* spans, int stride, uint32_t* stats, char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        finalize_device_model(m, build_fused(m));  // what gorp_engine_create does
        if (g_force_minimise)
            for (Tdfa& t : m.tdfas) minimise_tdfa(t);
        if (stats) {
            stats[0] = m.dfa.n_states;
            stats[1] = m.dfa.n_classes;
            stats[2] = m.symbols.n_classes;
            uint32_t ts = 0, tr = 0;
            for (auto& t : m.tdfas) {
                ts = std::max(ts, t.n_states);
                tr = std::max(tr, t.n_regs);
            }
            stats[3] = ts;
            stats[4] = tr;
        }
        const uint32_t C = m.dfa.n_classes;
        for (int64_t l = 0; l < n; ++l) {
            const uint16_t* u = text + starts[l];
            const int64_t L = ends[l] - starts[l];
            int32_t st = 0;
            for (int64_t i = 0; i < L && st >= 0; ++i) st = m.dfa.trans[static_cast<size_t>(st) * C + m.dfa.classmap[u[i]]];
            int32_t e = st < 0 ? -1 : m.dfa.accept_first[st];
            ext[l] = e;
            for (int k = 0; k < stride; ++k) spans[l * stride + k] = -1;
            if (e < 0) continue;
            const Tdfa& t = m.tdfas[e];
            std::vector<int32_t> regs(t.n_regs + 1, -7);
            uint32_t s = 0;
            bool ok = true;
            for (int64_t i = 0; i < L; ++i) {
                uint32_t k = m.symbols.classmap[u[i]];
                if ((u[i] & 0xFC00) == 0xD800 && i + 1 < L && (u[i + 1] & 0xFC00) == 0xDC00) k = m.symbols.pair_hi_class;
                uint32_t ent = t.trans[static_cast<size_t>(s) * t.n_classes + k];
                uint32_t nx = ent & 0xFFFF;
                if (nx == 0xFFFF) {
                    ok = false;
                    break;
                }
                uint32_t ol = ent >> 16;
                for (uint32_t q = t.op_off[ol]; q < t.op_off[ol + 1]; ++q) {
                    uint32_t op = t.ops[q], src = op & 0xFF;
                    regs[op >> 8] = src == 0xFF ? static_cast<int32_t>(i) : regs[src];
                }
                s = nx;
            }
            if (ok) ok = t.accepting[s] != 0;
            if (!ok) {
                ext[l] = -2 - e;
                if (m.pike_only[e]) {  // the simulated Pike VM decides (kernels/pike.cu, same loop)
                    const PikeTables& P = m.pike[e];
                    const uint32_t ent = 1 + P.n_slots;
                    std::vector<int32_t> lists[2];
                    lists[0].assign(static_cast<size_t>(P.n_insts) * ent, -1);
                    lists[1] = lists[0];
                    std::vector<uint32_t> seen(P.n_insts, 0);
                    uint32_t gen = 0, n_cur = 1;
                    int cur = 0;
                    lists[0][0] = 0;
                    for (int64_t p = 0; p < L && n_cur; ++p) {
                        uint32_t c = m.symbols.classmap[u[p]];
                        if ((u[p] & 0xFC00) == 0xD800 && p + 1 < L && (u[p + 1] & 0xFC00) == 0xDC00) c = m.symbols.pair_hi_class;
                        ++gen;
                        uint32_t n_nxt = 0;
                        const std::vector<int32_t>& from = lists[cur];
                        std::vector<int32_t>& to = lists[cur ^ 1];
                        for (uint32_t i = 0; i < n_cur; ++i) {
                            const int32_t pc = from[i * ent];
                            for (uint32_t j = P.clo_off[pc]; j < P.clo_off[pc + 1]; ++j) {
                                const int32_t tg = P.clo_target[j];
                                if (tg < 0 || seen[tg] == gen) continue;
                                seen[tg] = gen;
                                if (!P.accepts[static_cast<size_t>(tg) * P.n_classes + c]) continue;
                                to[n_nxt * ent] = tg + 1;
                                for (uint32_t k = 0; k < P.n_slots; ++k)
                                    to[n_nxt * ent + 1 + k] = (P.clo_mask[j] >> k) & 1 ? static_cast<int32_t>(p) : from[i * ent + 1 + k];
                                ++n_nxt;
                            }
                        }
                        cur ^= 1;
                        n_cur = n_nxt;
                    }
                    bool matched = false;
                    for (uint32_t i = 0; i < n_cur && !matched; ++i) {
                        const int32_t pc = lists[cur][i * ent];
                        for (uint32_t j = P.clo_off[pc]; j < P.clo_off[pc + 1]; ++j) {
                            if (P.clo_target[j] >= 0) continue;
                            for (uint32_t k = 0; k < P.n_slots && static_cast<int>(k) < stride; ++k)
                                spans[l * stride + k] = (P.clo_mask[j] >> k) & 1 ? static_cast<int32_t>(L) : lists[cur][i * ent + 1 + k];
                            matched = true;
                            break;
                        }
                    }
                    if (matched) ext[l] = e;
                }
                continue;
            }
            for (uint32_t k = 0; k < t.n_slots && static_cast<int>(k) < stride; ++k) {
                uint8_t f = t.fin[static_cast<size_t>(s) * t.n_slots + k];
                spans[l * stride + k] = f == 0xFF ? -1 : (f == 0xFE ? static_cast<int32_t>(L) : regs[f]);
            }
        }
        return 0;
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// The one-pass automaton (host/fused.hpp) interpreted one unit at a time: one table lookup per unit,
// "last position" per op slot, group boundaries resolved from the outcome at end of line.
// stats: [0] available, [1] states, [2] joint classes, [3] op slots, [4] outcomes. Returns 1 when not available.
extern "C" int ht_run_fused(const void* blob, size_t len, const uint16_t* text, const int64_t* starts, const int64_t* ends,
                            int64_t n, int32_t* ext, int32_t* spans, int stride, uint32_t* stats, char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        FusedAutomaton A = build_fused(m);
        if (stats) {
            stats[0] = A.available;
            stats[1] = A.n_states;
            stats[2] = A.n_jcls;
            stats[3] = A.n_op_slots;
            stats[4] = static_cast<uint32_t>(A.outcomes.size());
            uint32_t multi = 0;
            for (uint32_t r : A.res) multi += (r >> 8) != 0;
            stats[5] = multi;  // group boundaries with more than one writer slot
            stats[6] = static_cast<uint32_t>(A.res.size());
        }
        if (!A.available) {
            std::snprintf(err, errlen, "%s", A.why_not.c_str());
            return 1;
        }
        const uint32_t J = A.n_jcls;
        std::vector<int32_t> last(A.n_op_slots + 1);
        for (int64_t l = 0; l < n; ++l) {
            const uint16_t* u = text + starts[l];
            const int64_t L = ends[l] - starts[l];
            for (int k = 0; k < stride; ++k) spans[l * stride + k] = -1;
            std::fill(last.begin(), last.end(), -1);
            uint32_t st = 0;
            bool dead = false;
            for (int64_t i = 0; i < L; ++i) {
                uint32_t j = A.jcls[u[i]];
                if ((u[i] & 0xFC00) == 0xD800 && i + 1 < L && (u[i + 1] & 0xFC00) == 0xDC00) j = A.pair_of[j];
                const uint32_t ent = A.trans[static_cast<size_t>(st) * J + j];
                if ((ent & 0xFFFF) == 0xFFFF) {
                    dead = true;
                    break;
                }
                if (ent >> 16) last[ent >> 16] = static_cast<int32_t>(i);
                st = ent & 0xFFFF;
            }
            const FusedAutomaton::Outcome& o = A.outcomes[dead ? 0 : A.outcome_of[st]];
            ext[l] = o.ext_code;
            if (o.ext_code < 0) continue;
            const uint32_t ns = 2 * m.n_groups[o.ext_code];
            for (uint32_t k = 0; k < ns && static_cast<int>(k) < stride; ++k) {
                uint32_t packed = A.res[o.res_off + k];
                int32_t v = -1;
                for (; packed; packed >>= 8) {
                    const uint32_t id = packed & 0xFF;
                    v = std::max(v, id == FusedAutomaton::kLenSlot ? static_cast<int32_t>(L) : last[id]);
                }
                spans[l * stride + k] = v;
            }
        }
        return 0;
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// per-extraction capture automaton sizes: out[4*e..] = states, classes, registers, slots. Returns the extraction count.
extern "C" int ht_tdfa_sizes(const void* blob, size_t len, uint32_t* out, int cap, char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        finalize_device_model(m, build_fused(m));
        int n = 0;
        for (auto& t : m.tdfas) {
            if (n < cap) {
                out[4 * n] = t.n_states;
                out[4 * n + 1] = t.n_classes;
                out[4 * n + 2] = t.n_regs;
                out[4 * n + 3] = t.n_slots;
            }
            ++n;
        }
        return n;
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// the compacted combined DFA (host/automata.hpp: CompactDfa): trans[S*C] (-1 dead) and accept_first[S]. Returns S, sets *n_classes.
extern "C" int ht_compact_dfa(const void* blob, size_t len, int32_t* trans, int64_t cap, int32_t* accept_first, uint32_t* n_classes,
                              char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        *n_classes = m.dfa.n_classes;
        const int64_t n = static_cast<int64_t>(m.dfa.n_states) * m.dfa.n_classes;
        if (trans && n <= cap) {
            std::memcpy(trans, m.dfa.trans.data(), n * sizeof(int32_t));
            std::memcpy(accept_first, m.dfa.accept_first.data(), m.dfa.n_states * sizeof(int32_t));
        }
        return static_cast<int>(m.dfa.n_states);
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// The big-definition text path interpreted the way kernels/dfawalk.cu (K2b) and kernels/capwalk.cu (K4b) run it:
// '\n' split, combined DFA over the class-indexed table with SKIP / DEADSCAN / FIN rows in 16-unit blocks starting at
// the aligned block that holds the line start, then the capture walk over the extraction's table image (smem_variant:
// ids beyond DEAD read the DEAD row and the highest id seen survives; otherwise the physical FRZ rows), SLOW blocks
// replayed through the general tables. Returns the line count, or -1 (err) / -2 (tables not available).
#include "../../gorp_b200/csrc/host/walktables.hpp"

extern "C" int64_t ht_run_walk(const void* blob, size_t len, const uint16_t* text, int64_t n_units, int smem_variant, int64_t cap_lines,
                               int32_t* ext, int32_t* spans, int stride, char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        finalize_device_model(m, build_fused(m));
        const DfaWalkTable D = build_dfawalk_table(m);
        const CapImage I = build_cap_image(m, 4096);
        if (!D.available || !I.available) return -2;
        auto unit = [&](int64_t p) -> uint32_t { return p < n_units ? text[p] : 0x0Au; };
        int64_t n_lines = 0, a = 0;
        while (a < n_units) {
            int64_t b = a;
            while (b < n_units && text[b] != 0x0A) ++b;  // line = [a, b), its '\n' at b (virtual at n_units)
            if (n_lines >= cap_lines) return -1;
            // ---- DFA
            int64_t q = a & ~int64_t(15);
            uint32_t st = a - q ? D.n_states + static_cast<uint32_t>(a - q) : 0u;
            while (st < D.fin_base) {
                for (int k = 0; k < 16; ++k) {
                    const uint32_t u = unit(q + k);
                    const uint32_t col = u < 128 ? D.cls128[u] / 2u : D.xcls[u];
                    st = D.rows[static_cast<size_t>(st) * D.K + col];
                }
                q += 16;
            }
            const int32_t e = static_cast<int32_t>(st - D.fin_base) - 1;
            int32_t* out = spans + n_lines * stride;
            for (int k = 0; k < stride; ++k) out[k] = -1;
            ext[n_lines] = e;
            if (e >= 0) {
                // ---- capture
                const CapImageExt& fx = I.ext[e];
                const Tdfa& t = m.tdfas[e];
                std::vector<int32_t> regs(I.n_regs + 1, -7);
                const uint32_t S = fx.n_states, Cn = m.symbols.n_classes;
                q = a & ~int64_t(15);
                uint32_t cs = a - q ? (S + static_cast<uint32_t>(a - q) - 1) * fx.row_bytes : 0u;
                while (cs < fx.dead_off) {
                    const uint32_t st0 = cs;
                    uint32_t fin = 0;
                    for (int k = 0; k < 16; ++k) {
                        const uint32_t u = unit(q + k);
                        uint32_t c4;
                        if (u < 128) {
                            c4 = I.cls128[u];
                        } else {
                            c4 = 4u * m.symbols.classmap[u];
                            if ((u & 0xFC00u) == 0xD800u && (unit(q + k + 1) & 0xFC00u) == 0xDC00u) c4 = 4u * m.symbols.pair_hi_class;
                        }
                        const uint32_t row = smem_variant ? std::min(cs, fx.dead_off) : cs;
                        const uint32_t ent = I.image[(fx.tab_off + row + c4) / 4];
                        cs = ent >> 6;
                        fin = std::max(fin, cs);
                        regs[ent & 63u] = static_cast<int32_t>(q + k - a);
                    }
                    if (smem_variant && fin >= fx.dead_off) cs = fin;
                    if (cs == fx.slow_off) {  // replay the block through the general tables (kernels/capwalk.cu: cw_slow16)
                        uint32_t row = st0 / fx.row_bytes;
                        for (int k = 0; k < 16; ++k) {
                            if (row >= S + 15) break;
                            const int64_t p = q + k;
                            const uint32_t u = unit(p);
                            if (row >= S) {
                                row = row == S ? 0u : row - 1;
                                continue;
                            }
                            if (u == 0x0A) {
                                row = S + 17 + row;
                                break;
                            }
                            uint32_t sym = m.symbols.classmap[u];
                            if ((u & 0xFC00u) == 0xD800u && p + 1 < n_units && (text[p + 1] & 0xFC00u) == 0xDC00u) sym = m.symbols.pair_hi_class;
                            const uint32_t ent = t.trans[static_cast<size_t>(row) * Cn + sym];
                            if ((ent & 0xFFFFu) == 0xFFFFu) {
                                row = S + 15;
                                continue;
                            }
                            const uint32_t ol = ent >> 16;
                            for (uint32_t i = t.op_off[ol]; i < t.op_off[ol + 1]; ++i) {
                                const uint32_t op = t.ops[i], src = op & 0xFFu;
                                regs[op >> 8] = src == 0xFFu ? static_cast<int32_t>(p - a) : regs[src];
                            }
                            row = ent & 0xFFFFu;
                        }
                        cs = row * fx.row_bytes;
                    }
                    q += 16;
                }
                bool ok = cs >= fx.frz_off;
                uint32_t s = 0;
                if (ok) {
                    s = (cs - fx.frz_off) / fx.row_bytes;
                    ok = t.accepting[s] != 0;
                }
                if (!ok) {
                    ext[n_lines] = -2 - e;
                } else {
                    for (uint32_t k = 0; k < t.n_slots && static_cast<int>(k) < stride; ++k) {
                        const uint8_t f = t.fin[static_cast<size_t>(s) * t.n_slots + k];
                        out[k] = f == 0xFF ? -1 : (f == 0xFE ? static_cast<int32_t>(b - a) : regs[f]);
                    }
                }
            }
            ++n_lines;
            a = b + 1;
        }
        return n_lines;
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// Tail automata (host/tails.hpp): per extraction out[4*e..] = available, states, op slots, outcomes; summary[0..4] = width,
// cut states, compact DFA states, any. Returns the extraction count.
#include "../../gorp_b200/csrc/host/tails.hpp"

extern "C" int ht_tail_sizes(const void* blob, size_t len, uint32_t* out, int cap, uint32_t* summary, char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        finalize_device_model(m, build_fused(m));
        const TailSet T = build_tails(def, m);
        int n = 0;
        for (auto& t : T.tails) {
            if (n < cap) {
                out[4 * n] = t.available ? 1u : 0u;
                out[4 * n + 1] = t.n_states;
                out[4 * n + 2] = t.n_op_slots;
                out[4 * n + 3] = static_cast<uint32_t>(t.outcomes.size());
            }
            if (!t.available && n < 3) std::snprintf(err, errlen, "tail %d: %s", n, t.why_not.c_str());
            ++n;
        }
        summary[0] = T.width;
        summary[1] = T.n_cut_states;
        summary[2] = m.dfa.n_states;
        summary[3] = T.any ? 1u : 0u;
        return n;
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// The big-definition text path with the early-exit cut (host/tails.hpp) interpreted the way kernels/dfawalk.cu (K2b over
// the cut table) and kernels/tailwalk.cu (K4c over the tail image) run it: '\n' split; combined DFA over the cut table in
// 16-unit blocks until a FIN row (dead => MISS at once, cut state => candidate e); tail automaton of the candidate from the
// line start, op slots hold position + 1, outcome + recipes at the end. Lines whose candidate has no tail fall back to the
// capture automaton of the extraction (general tables) — those extractions are never cut, so the candidate is exact.
// Returns the line count, or -1 (err) / -2 (no tails). stats[0] = lines that left the DFA walk early, [1] = units walked by
// the DFA, [2] = cut-table states, [3] = lines decided by a tail.
extern "C" int64_t ht_run_tails(const void* blob, size_t len, const uint16_t* text, int64_t n_units, int64_t cap_lines, int32_t* ext,
                                int32_t* spans, int stride, uint64_t* stats, char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        finalize_device_model(m, build_fused(m));
        const TailSet T = build_tails(def, m);
        if (!T.any) return -2;
        const DfaWalkTable D = build_dfawalk_table_cut(m, T.cut_of_state);
        const TailImage I = build_tail_image(T, static_cast<uint32_t>(stride));
        if (!D.available || !I.available) return -2;
        auto unit = [&](int64_t p) -> uint32_t { return p < n_units ? text[p] : 0x0Au; };
        if (stats) stats[0] = stats[1] = stats[3] = 0, stats[2] = D.n_states;
        int64_t n_lines = 0, a = 0;
        while (a < n_units) {
            int64_t b = a;
            while (b < n_units && text[b] != 0x0A) ++b;
            if (n_lines >= cap_lines) return -1;
            // ---- combined DFA, cut
            int64_t q = a & ~int64_t(15);
            uint32_t st = a - q ? D.n_states + static_cast<uint32_t>(a - q) : 0u;
            while (st < D.fin_base) {
                for (int k = 0; k < 16; ++k) {
                    const uint32_t u = unit(q + k);
                    const uint32_t col = u < 128 ? D.cls128[u] / 2u : D.xcls[u];
                    st = D.rows[static_cast<size_t>(st) * D.K + col];
                }
                q += 16;
            }
            if (stats) {
                stats[1] += static_cast<uint64_t>(std::min<int64_t>(q, b + 1) - a);
                if (q <= b) ++stats[0];
            }
            const int32_t e = static_cast<int32_t>(st - D.fin_base) - 1;
            int32_t* out = spans + n_lines * stride;
            for (int k = 0; k < stride; ++k) out[k] = -1;
            ext[n_lines] = e;
            if (e >= 0 && I.ext[e].available) {
                if (stats) ++stats[3];
                const TailImageExt& x = I.ext[e];
                const uint16_t* tab = I.image.data() + x.tab_off / 2;
                std::vector<uint32_t> slots(64, 0xDEAD);  // garbage on purpose: only the init slots are reset per line
                for (uint32_t i = 0; i < x.n_init; ++i) slots[I.init_slots[x.init_off + i]] = 0;
                q = a & ~int64_t(15);
                uint32_t row = a - q ? x.n_states + static_cast<uint32_t>(a - q) - 1 : 0u;
                while (row < x.fin_base) {
                    for (int k = 0; k < 16; ++k) {
                        const uint32_t u = unit(q + k);
                        uint32_t col = u < 128 ? u : T.xcol[u];
                        if ((u & 0xFC00u) == 0xD800u && (unit(q + k + 1) & 0xFC00u) == 0xDC00u) col = T.pair_col[col];
                        const uint32_t ent = tab[static_cast<size_t>(row) * I.width + col];
                        row = ent >> 6;
                        slots[ent & 63u] = static_cast<uint32_t>(q + k - a + 1);
                    }
                    q += 16;
                }
                const uint32_t o = row - x.fin_base;
                const int32_t code = I.oext[x.oext_off + o];
                ext[n_lines] = code;
                if (code >= 0)
                    for (int k = 0; k < stride; ++k) {
                        uint32_t rec = I.res[x.res_off + static_cast<size_t>(o) * stride + k];
                        int32_t val = -1;
                        if (rec == 0xFF) {
                            val = static_cast<int32_t>(b - a);
                        } else if (rec) {
                            uint32_t best = 0;
                            for (; rec; rec >>= 8) best = std::max(best, slots[rec & 0xFFu]);
                            val = static_cast<int32_t>(best) - 1;
                        }
                        out[k] = val;
                    }
            } else if (e >= 0) {  // no tail: the general capture automaton (as ht_run)
                const Tdfa& t = m.tdfas[e];
                std::vector<int32_t> regs(t.n_regs + 1, -7);
                uint32_t s = 0;
                bool ok = true;
                const int64_t L = b - a;
                for (int64_t i = 0; i < L; ++i) {
                    const uint32_t u = text[a + i];
                    uint32_t k = m.symbols.classmap[u];
                    if ((u & 0xFC00) == 0xD800 && i + 1 < L && (text[a + i + 1] & 0xFC00) == 0xDC00) k = m.symbols.pair_hi_class;
                    const uint32_t ent = t.trans[static_cast<size_t>(s) * t.n_classes + k];
                    if ((ent & 0xFFFF) == 0xFFFF) {
                        ok = false;
                        break;
                    }
                    const uint32_t ol = ent >> 16;
                    for (uint32_t i2 = t.op_off[ol]; i2 < t.op_off[ol + 1]; ++i2) {
                        const uint32_t op = t.ops[i2], src = op & 0xFF;
                        regs[op >> 8] = src == 0xFF ? static_cast<int32_t>(i) : regs[src];
                    }
                    s = ent & 0xFFFF;
                }
                if (ok) ok = t.accepting[s] != 0;
                if (!ok) {
                    ext[n_lines] = -2 - e;
                } else {
                    for (uint32_t k = 0; k < t.n_slots && static_cast<int>(k) < stride; ++k) {
                        const uint8_t f = t.fin[static_cast<size_t>(s) * t.n_slots + k];
                        out[k] = f == 0xFF ? -1 : (f == 0xFE ? static_cast<int32_t>(L) : regs[f]);
                    }
                }
            }
            ++n_lines;
            a = b + 1;
        }
        return n_lines;
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// The fused walk (small definitions): the one-pass automaton as ONE tail table (host/tails.hpp: build_fused_tailset) walked by
// every line [starts[i], ends[i]) the way kernels/tailwalk.cu walks it in "all" mode: state 0, one lookup per unit (a unit
// >= 0x80 through the column map, a surrogate pair through pair_col, a '\n' inside the line — List<String> form — through
// nl_data_col), the terminator column at the end of the line, op slots hold position + 1, outcome row -> ext code + recipes.
// Returns 0, 1 (not available) or -1 (err).
extern "C" int ht_run_fused_tail(const void* blob, size_t len, const uint16_t* text, const int64_t* starts, const int64_t* ends, int64_t n,
                                 int32_t* ext, int32_t* spans, int stride, char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        const FusedAutomaton F = build_fused(m);
        finalize_device_model(m, F);
        if (!F.available) {
            std::snprintf(err, errlen, "%s", F.why_not.c_str());
            return 1;
        }
        const TailSet T = build_fused_tailset(F, m, static_cast<uint32_t>(stride));
        const TailImage I = build_tail_image(T, static_cast<uint32_t>(stride));
        if (!I.available || !I.ext[0].available) {
            std::snprintf(err, errlen, "the fused automaton does not fit the tail image limits");
            return 1;
        }
        const TailImageExt& x = I.ext[0];
        const uint16_t* tab = I.image.data() + x.tab_off / 2;
        for (int64_t i = 0; i < n; ++i) {
            const int64_t a = starts[i], b = ends[i];
            std::vector<uint32_t> slots(64, 0xDEAD);  // garbage on purpose: only the init slots are reset per line
            for (uint32_t k = 0; k < x.n_init; ++k) slots[I.init_slots[x.init_off + k]] = 0;
            uint32_t row = 0;
            for (int64_t p = a; p <= b && row < x.fin_base; ++p) {
                uint32_t col = 0x0Au;  // the terminator
                if (p < b) {
                    const uint32_t u = text[p];
                    col = u == 0x0Au ? T.nl_data_col : (u < 128 ? u : T.xcol[u]);
                    if ((u & 0xFC00u) == 0xD800u && p + 1 < b && (text[p + 1] & 0xFC00u) == 0xDC00u) col = T.pair_col[col];
                }
                const uint32_t ent = tab[static_cast<size_t>(row) * I.width + col];
                row = ent >> 6;
                slots[ent & 63u] = static_cast<uint32_t>(p - a + 1);
            }
            const uint32_t o = row - x.fin_base;
            const int32_t code = I.oext[x.oext_off + o];
            ext[i] = code;
            int32_t* out = spans + i * stride;
            for (int k = 0; k < stride; ++k) {
                uint32_t rec = I.res[x.res_off + static_cast<size_t>(o) * stride + k];
                int32_t val = -1;
                if (code >= 0 && rec == 0xFF) {
                    val = static_cast<int32_t>(b - a);
                } else if (code >= 0 && rec) {
                    uint32_t best = 0;
                    for (; rec; rec >>= 8) best = std::max(best, slots[rec & 0xFFu]);
                    val = static_cast<int32_t>(best) - 1;
                }
                out[k] = val;
            }
        }
        return 0;
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}

// Which side of each table limit a definition lands on (the choices engine.cu makes when it builds an engine, minus the
// shared-memory budgets, which depend on the kernels' launch shapes). out[0..11] = largest tag-register count of the capture
// automata, span stride (2 x the most groups), fused automaton available, its op slots, its outcomes, its several-writer
// group boundaries, fused-walk table image available, its table bytes, capture image (K4b) available, fast capture image
// (K4 fast) available, tails of any extraction, extractions that fall back to the Pike VM. tail[e] = the tail image of
// extraction e is available. Returns the extraction count, or -1 (err).
extern "C" int ht_layout(const void* blob, size_t len, uint32_t* out, uint8_t* tail, int cap, char* err, int errlen) {
    try {
        CompiledDefinition def = parse_blob(blob, len);
        DeviceModel m = build_device_model(def);
        const FusedAutomaton F = build_fused(m);
        finalize_device_model(m, F);
        const size_t E = m.n_groups.size();
        uint32_t max_regs = 0, max_groups = 0, n_pike = 0;
        for (const Tdfa& t : m.tdfas) max_regs = std::max(max_regs, t.n_regs);
        for (uint32_t g : m.n_groups) max_groups = std::max(max_groups, g);
        for (uint8_t p : m.pike_only) n_pike += p ? 1u : 0u;
        const uint32_t stride = 2 * max_groups;
        std::fill(out, out + 12, 0u);
        out[0] = max_regs;
        out[1] = stride;
        out[2] = F.available ? 1u : 0u;
        if (F.available) {
            out[3] = F.n_op_slots;
            out[4] = static_cast<uint32_t>(F.outcomes.size());
            for (uint32_t r : F.res) out[5] += r >= 256u ? 1u : 0u;
            if (stride > 0) {
                const TailImage I = build_tail_image(build_fused_tailset(F, m, stride), stride);
                out[6] = I.available && I.ext[0].available ? 1u : 0u;
                out[7] = I.max_table_bytes;
            }
        }
        out[8] = build_cap_image(m, 4096).available ? 1u : 0u;
        // engine.cu, fast tier image: every table within 16-bit row offsets, image + registers within 160 KB
        {
            const uint32_t row_bytes = (m.symbols.n_classes + 1) * 4;
            size_t words = 128;
            bool ok = true;
            for (const Tdfa& t : m.tdfas) {
                const uint64_t rows = 2ull * t.n_states + 9;
                ok = ok && rows * row_bytes <= 0xFFFC;
                words += rows * (row_bytes / 4);
            }
            words = (words + 3) & ~size_t(3);
            const size_t reg_stride = 512 * 4;  // kernels.cuh: kCapFastThreads x 4
            out[9] = ok && words * 4 + (max_regs + 2) * reg_stride <= 160 * 1024 && (max_regs + 2) * reg_stride <= 0x10000 ? 1u : 0u;
        }
        const TailSet T = build_tails(def, m);
        out[10] = T.any ? 1u : 0u;
        out[11] = n_pike;
        const TailImage TI = build_tail_image(T, stride);
        for (size_t e = 0; e < E && static_cast<int>(e) < cap; ++e) tail[e] = T.any && TI.ext[e].available ? 1u : 0u;
        return static_cast<int>(E);
    } catch (const std::exception& e) {
        std::snprintf(err, errlen, "%s", e.what());
        return -1;
    }
}
