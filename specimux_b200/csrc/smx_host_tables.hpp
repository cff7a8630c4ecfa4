// smx_host_tables.hpp -- host-side construction of the match tables (shared by the CUDA API and
// the CPU kernel simulator used in unit tests).  Builds IUPAC-aware Peq masks with edlib's
// additionalEqualities semantics (reference: constants.py:13-20, alignment.py:42) and the
// (b1, b2) -> specimen rows lookup (databases.py:219-245).
#pragma once
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "smx_core.cuh"
#include "smx_pack.cuh"     // read_code / read_code_rc, the read encoding

namespace smx {

static const char kCodes[] = "ACGTRYSWKMBDHVN";

inline int code_of(char ch) {
    const char *p = strchr(kCodes, ch);
    return (p && ch) ? (int)(p - kCodes) : -1;
}

// base set of an IUPAC code as a 4-bit mask over A,C,G,T (constants.py:13-20)
inline int base_set(int code) {
    static const int sets[15] = {1, 2, 4, 8, 1 | 4, 2 | 8, 2 | 4, 1 | 8, 4 | 8, 1 | 2,
                                 2 | 4 | 8, 1 | 4 | 8, 1 | 2 | 8, 1 | 2 | 4, 15};
    return sets[code];
}

// edlib additionalEqualities semantics: a == b, or (code, base) listed in either order.
inline bool sym_equal(int pat, int rd) {
    if (rd == kSymOther) return false;
    if (pat == rd) return true;
    if (pat >= 4 && rd < 4) return (base_set(pat) >> rd) & 1;
    if (rd >= 4 && pat < 4) return (base_set(rd) >> pat) & 1;
    return false;
}

// Multi-word Peq of a long pattern: row i sits at bit (32*sw - m + i) of a 32*sw-bit vector, word w
// of symbol c at out[c * sw + w].
inline bool build_peq_long(const char *s, int m, bool reversed, int sw, u32 *out /*16*sw*/) {
    for (int i = 0; i < 16 * sw; ++i) out[i] = 0;
    for (int i = 0; i < m; ++i) {
        int pc = code_of(s[reversed ? m - 1 - i : i]);
        if (pc < 0) return false;
        int pos = 32 * sw - m + i;
        for (int c = 0; c < 16; ++c)
            if (sym_equal(pc, c)) out[c * sw + (pos >> 5)] |= 1u << (pos & 31);
    }
    return true;
}

inline bool build_peq(const char *s, int m, bool reversed, u64 *out /*16*/) {
    for (int c = 0; c < 16; ++c) out[c] = 0;
    for (int i = 0; i < m; ++i) {
        int pc = code_of(s[reversed ? m - 1 - i : i]);
        if (pc < 0) return false;
        for (int c = 0; c < 16; ++c)
            if (sym_equal(pc, c)) out[c] |= 1ull << (64 - m + i);
    }
    return true;
}


struct HostTables {
    Tables t;
    std::vector<u64> peq_rc, peq_rcrev, peq_fw, spec_key, spec_p1, spec_p2;
    std::vector<unsigned char> b_len, bw_len, bw_primer, b_codes;
    std::vector<u32> b_code_off, bw_iupac;
    std::vector<u32> pb_barcode, pair_fwd, pair_rev, spec_key_off, spec_row, bw_row, bw_valid, beq;
    std::vector<unsigned short> bw_list;
    std::vector<unsigned short> bt_g0, bt_class_tasks;     // stage-2 tasks; task ids grouped by (words per task, barcode length)
    std::vector<unsigned char> bt_nw;
    std::vector<u32> bt_row, bt_eq, bt_quad;
    std::vector<i32> bt_quad_row;
    std::vector<BtClass> bt_classes;                       // one kernel launch each
    std::vector<i32> pair_pool, spec_pool, spec_dense;
    std::vector<u32> peq_long;
    std::vector<unsigned char> prow_code;      // [primer][32] IUPAC code of primer_rc row i (sliced primer search)
    int max_nb = 0;
    std::string error;

    bool err(const char *fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        error = buf;
        return false;
    }

    // Validates and builds everything; on success `t` holds HOST pointers into the vectors.
    bool build(const smx_tables *tb, const smx_params *pr) {
        if (!tb || !pr) return err("null argument");
        if (tb->n_primers == 0 || tb->n_primers > SMX_MAX_PRIMERS)
            return err("n_primers=%u outside 1..%d", tb->n_primers, SMX_MAX_PRIMERS);
        if (tb->n_pairs > (uint32_t)kMaxPairs) return err("%u primer pairs exceed the supported %d", tb->n_pairs, kMaxPairs);
        if (pr->search_len < 1 || pr->search_len > SMX_MAX_SEARCH_LEN)
            return err("search_len=%d outside 1..%d", pr->search_len, SMX_MAX_SEARCH_LEN);
        if (pr->trim < SMX_TRIM_NONE || pr->trim > SMX_TRIM_TAILS) return err("bad trim mode");
        memset(&t, 0, sizeof(t));
        const int nP = (int)tb->n_primers;
        t.n_primers = nP; t.n_pairs = (int)tb->n_pairs; t.n_specimens = (int)tb->n_specimens;
        t.L = pr->search_len; t.wpw = (t.L + 7) / 8; t.mw = (t.L + 31) / 32; t.nw2 = (t.L + 15) / 16;
        t.k_idx = pr->max_dist_index; t.blen_max = pr->barcode_length;
        t.preorient = pr->preorient != 0; t.prefilter = pr->prefilter != 0; t.trim = pr->trim;
        t.derep_best = pr->dereplicate_best != 0; t.min_length = pr->min_length; t.max_length = pr->max_length;
        if (t.k_idx < 0) return err("negative barcode distance threshold");

        peq_rc.assign((size_t)nP * 16, 0); peq_rcrev.assign((size_t)nP * 16, 0); peq_fw.assign((size_t)nP * 16, 0);
        peq_long.clear();
        prow_code.assign((size_t)nP * 32, 0);
        for (int p = 0; p < nP; ++p) {
            int m = (int)(tb->primer_off[p + 1] - tb->primer_off[p]);
            if (m < 1 || m > SMX_MAX_LONG_PATTERN) return err("primer %d length %d outside 1..%d", p, m, SMX_MAX_LONG_PATTERN);
            int k = tb->primer_k[p];
            if (k < 0 || k >= m) return err("primer %d max distance %d must be in [0, length %d)", p, k, m);
            if (k > 127) return err("primer %d max distance %d exceeds 127 (smx_record.dist is 8 bits)", p, k);
            t.p_len[p] = (unsigned short)m; t.p_k[p] = (short)k; t.p_dir[p] = tb->primer_dir[p];
            t.p_fidx[p] = tb->primer_file_index[p];
            if (m > 32) t.use64 = 1;
            t.p_sw[p] = 0; t.p_long[p] = -1;
            if (m > SMX_MAX_PATTERN) {
                // warp-cooperative multi-word search: lanes per problem = the narrowest segment width >= ceil(m/32)
                // that gives a different number of reads per warp (3 -> 10 reads, 4 -> 8, 5 -> 6, 6 -> 5, 8 -> 4,
                // 10 -> 3, 16 -> 2, 32 -> 1)
                const int words = (m + 31) / 32;
                static const int kWidths[] = {3, 4, 5, 6, 8, 10, 16, 32};
                int sw = 32;
                for (int w : kWidths) if (w >= words) { sw = w; break; }
                t.p_sw[p] = (unsigned char)sw; t.p_long[p] = (int)peq_long.size();
                size_t base = peq_long.size();
                peq_long.resize(base + (size_t)3 * 16 * sw, 0);
                if (!build_peq_long(tb->primer_rc + tb->primer_off[p], m, false, sw, &peq_long[base]) ||
                    !build_peq_long(tb->primer_rc + tb->primer_off[p], m, true, sw, &peq_long[base + (size_t)16 * sw]) ||
                    !build_peq_long(tb->primer_seq + tb->primer_off[p], m, false, sw, &peq_long[base + (size_t)32 * sw]))
                    return err("primer %d has a non-IUPAC character", p);
                t.pb_off[p] = tb->pb_off[p];
                continue;
            }
            if (!build_peq(tb->primer_rc + tb->primer_off[p], m, false, &peq_rc[(size_t)p * 16]) ||
                !build_peq(tb->primer_rc + tb->primer_off[p], m, true, &peq_rcrev[(size_t)p * 16]) ||
                !build_peq(tb->primer_seq + tb->primer_off[p], m, false, &peq_fw[(size_t)p * 16]))
                return err("primer %d has a non-IUPAC character", p);
            for (int i = 0; i < m && i < 32; ++i) prow_code[(size_t)p * 32 + i] = (unsigned char)code_of(tb->primer_rc[tb->primer_off[p] + i]);
            t.pb_off[p] = tb->pb_off[p];
        }
        t.pb_off[nP] = tb->pb_off[nP];
        t.sliced = !t.use64;
        if (peq_long.empty()) peq_long.push_back(0);
        t.peq_long = peq_long.data();
        const u32 n_list = tb->pb_off[nP];
        std::vector<std::string> b_str(n_list);
        b_len.assign(n_list, 0);
        pb_barcode.assign(tb->pb_barcode, tb->pb_barcode + n_list);
        max_nb = 0;
        for (int p = 0; p < nP; ++p) {
            int nb = (int)(tb->pb_off[p + 1] - tb->pb_off[p]);
            max_nb = std::max(max_nb, nb);
            bool fwd = tb->primer_dir[p] == 0;
            for (u32 e = tb->pb_off[p]; e < tb->pb_off[p + 1]; ++e) {
                u32 id = tb->pb_barcode[e];
                if (id >= (fwd ? tb->n_b1 : tb->n_b2)) return err("barcode id out of range");
                const u32 *off = fwd ? tb->b1_off : tb->b2_off;
                const char *s = (fwd ? tb->b1_rc : tb->b2_rc) + off[id];
                int m = (int)(off[id + 1] - off[id]);
                if (m < 1 || m + t.k_idx > SMX_MAX_PATTERN)
                    return err("barcode length %d + k %d exceeds %d", m, t.k_idx, SMX_MAX_PATTERN);
                if (t.k_idx >= m) return err("barcode distance threshold %d must be below barcode length %d", t.k_idx, m);
                for (int i = 0; i < m; ++i) if (code_of(s[i]) < 0) return err("barcode has a non-IUPAC character");
                b_str[e].assign(s, s + m);
                b_len[e] = (unsigned char)m;
            }
        }
        b_codes.clear(); b_code_off.assign(n_list + 1, 0);
        for (u32 e = 0; e < n_list; ++e) {
            b_code_off[e] = (u32)b_codes.size();
            for (char ch : b_str[e]) b_codes.push_back((unsigned char)code_of(ch));
        }
        b_code_off[n_list] = (u32)b_codes.size();
        if (b_codes.empty()) b_codes.push_back(0);
        // bit-sliced barcode words: per primer, barcodes grouped by length, 32 to a word
        bw_len.clear(); bw_primer.clear(); bw_row.clear(); bw_valid.clear(); bw_list.clear(); beq.clear(); bw_iupac.clear();
        for (int p = 0; p < nP; ++p) {
            t.bw_off[p] = (u32)bw_len.size();
            std::vector<int> lens;
            for (u32 e = tb->pb_off[p]; e < tb->pb_off[p + 1]; ++e) lens.push_back(b_len[e]);
            std::sort(lens.begin(), lens.end());
            lens.erase(std::unique(lens.begin(), lens.end()), lens.end());
            for (int m : lens) {
                std::vector<u32> members;
                for (u32 e = tb->pb_off[p]; e < tb->pb_off[p + 1]; ++e) if (b_len[e] == m) members.push_back(e);
                for (size_t base = 0; base < members.size(); base += 32) {
                    size_t cnt = std::min<size_t>(32, members.size() - base);
                    bw_len.push_back((unsigned char)m);
                    bw_primer.push_back((unsigned char)p);
                    bw_row.push_back((u32)(beq.size() / 16));
                    bw_valid.push_back(cnt == 32 ? ~0u : ((1u << cnt) - 1));
                    bw_iupac.push_back(0);
                    size_t row0 = beq.size();
                    beq.resize(row0 + (size_t)m * 16, 0);
                    for (size_t q = 0; q < 32; ++q) {
                        if (q >= cnt) { bw_list.push_back(0); continue; }
                        u32 e = members[base + q];
                        bw_list.push_back((unsigned short)(e - tb->pb_off[p]));
                        for (int i = 0; i < m; ++i) {
                            int pc = code_of(b_str[e][i]);
                            if (pc > 3) bw_iupac.back() |= 1u << q;
                            for (int c = 0; c < 16; ++c)
                                if (sym_equal(pc, c)) beq[row0 + (size_t)i * 16 + c] |= 1u << q;
                        }
                    }
                }
            }
        }
        t.bw_off[nP] = (u32)bw_len.size();
        t.n_bwords = (int)bw_len.size();
        t.hit_cap = 4;
        // stage-2 tasks: consecutive bwords of one primer and one length, up to kMaxTaskWords to a task (one word
        // when the flank does not fit the 16-column register form, or k is beyond the multi-word instantiations)
        bt_g0.clear(); bt_nw.clear(); bt_row.clear(); bt_eq.clear(); bt_class_tasks.clear(); bt_quad.clear(); bt_quad_row.clear();
        for (int p = 0; p < nP; ++p) {
            t.bt_off[p] = (u32)bt_g0.size();
            u32 g = t.bw_off[p];
            while (g < t.bw_off[p + 1]) {
                const int m = bw_len[g];
                const u32 max_words = (m + t.k_idx <= 16 && t.k_idx <= kMaxTaskK) ? (u32)kMaxTaskWords : 1u;
                u32 nw = 1;
                while (nw < max_words && g + nw < t.bw_off[p + 1] && bw_len[g + nw] == m) ++nw;
                const u32 S = nw == 1 ? 1u : nw == 2 ? 2u : 4u;
                bt_g0.push_back((unsigned short)g);
                bt_nw.push_back((unsigned char)nw);
                while (bt_eq.size() % 4) bt_eq.push_back(0);            // vector loads: 16-byte aligned tables
                bt_row.push_back((u32)bt_eq.size());
                const size_t base = bt_eq.size();
                bt_eq.resize(base + (size_t)m * 16 * S, 0);
                for (u32 q = 0; q < nw; ++q)
                    for (int i = 0; i < m; ++i)
                        for (int c = 0; c < 16; ++c)
                            bt_eq[base + ((size_t)i * 16 + c) * S + q] = beq[((size_t)bw_row[g + q] + i) * 16 + c];
                // narrow word (<= 8 barcodes, register form): the four-entries-to-a-word table, indexed per row by the
                // four entries' symbols (0..3 = A/C/G/T, 4 = beyond the flank: matches nothing), entry q in byte lane q
                bt_quad_row.push_back(-1);
                if (quad_enabled() && nw == 1 && m + t.k_idx <= 16 && t.k_idx <= kMaxTaskK && (bw_valid[g] & ~0xFFu) == 0) {
                    bt_quad_row.back() = (i32)bt_quad.size();
                    const size_t qb = bt_quad.size();
                    bt_quad.resize(qb + (size_t)m * kQuadRow, 0);
                    for (int i = 0; i < m; ++i)
                        for (int idx = 0; idx < kQuadRow; ++idx) {
                            u32 w = 0;
                            int rest = idx;
                            for (int q = 0; q < 4; ++q) {
                                const int sym = rest % kQuadSyms;
                                rest /= kQuadSyms;
                                if (sym < 4) w |= (beq[((size_t)bw_row[g] + i) * 16 + sym] & 0xFFu) << (8 * q);
                            }
                            bt_quad[qb + (size_t)i * kQuadRow + idx] = w;
                        }
                }
                g += nw;
            }
        }
        t.bt_off[nP] = (u32)bt_g0.size();
        t.n_btasks = (int)bt_g0.size();
        if (bt_g0.size() > 65535) return err("more than 65535 barcode tasks");
        bt_classes.clear();
        for (int w = 1; w <= kMaxTaskWords; ++w)
            for (int m = 1; m <= SMX_MAX_PATTERN; ++m) {
                for (int quad = 0; quad < 2; ++quad) {
                    BtClass c;
                    c.nw = w; c.m = m; c.quad = quad; c.off = (u32)bt_class_tasks.size(); c.count = 0;
                    for (size_t k = 0; k < bt_nw.size(); ++k)
                        if (bt_nw[k] == w && bw_len[bt_g0[k]] == m && (bt_quad_row[k] >= 0) == (quad != 0)) {
                            bt_class_tasks.push_back((unsigned short)k);
                            ++c.count;
                        }
                    if (c.count) bt_classes.push_back(c);
                }
            }
        if (bt_eq.empty()) bt_eq.push_back(0);
        if (bt_g0.empty()) { bt_g0.push_back(0); bt_nw.push_back(0); bt_row.push_back(0); bt_quad_row.push_back(-1); }
        if (bt_quad.empty()) bt_quad.push_back(0);
        if (bt_class_tasks.empty()) bt_class_tasks.push_back(0);
        for (int p = 0; p < nP; ++p)
            if (tb->pb_off[p + 1] - tb->pb_off[p] > 65535) return err("primer %d has more than 65535 barcodes", p);

        u32 run = 0;
        for (int s = 0; s < 2; ++s)
            for (int p = 0; p < nP; ++p) { t.bslot_base[s * nP + p] = run; run += tb->pb_off[p + 1] - tb->pb_off[p]; }
        t.total_bslots = (int)run;

        for (u32 i = 0; i < tb->n_pairs; ++i)
            if (tb->pair_fwd[i] >= (u32)nP || tb->pair_rev[i] >= (u32)nP) return err("pair index out of range");
        pair_fwd.assign(tb->pair_fwd, tb->pair_fwd + tb->n_pairs);
        pair_rev.assign(tb->pair_rev, tb->pair_rev + tb->n_pairs);
        pair_pool.assign(tb->pair_pool, tb->pair_pool + tb->n_pairs);

        // specimen lookup: rows grouped by (b1, b2), file order inside a group
        spec_row.resize(tb->n_specimens);
        for (u32 i = 0; i < tb->n_specimens; ++i) spec_row[i] = i;
        auto key_of = [&](u32 r) { return ((u64)tb->spec_b1[r] << 32) | tb->spec_b2[r]; };
        std::stable_sort(spec_row.begin(), spec_row.end(), [&](u32 a, u32 c) { return key_of(a) < key_of(c); });
        spec_key.clear(); spec_key_off.clear();
        for (u32 i = 0; i < tb->n_specimens; ++i) {
            u64 k = key_of(spec_row[i]);
            if (spec_key.empty() || spec_key.back() != k) { spec_key.push_back(k); spec_key_off.push_back(i); }
        }
        spec_key_off.push_back(tb->n_specimens);
        t.n_keys = (int)spec_key.size();
        t.n_b2 = (int)tb->n_b2;
        spec_dense.clear();
        if ((u64)tb->n_b1 * tb->n_b2 <= (4u << 20) && tb->n_b1 && tb->n_b2) {
            spec_dense.assign((size_t)tb->n_b1 * tb->n_b2, -1);
            for (size_t i = 0; i < spec_key.size(); ++i)
                spec_dense[(size_t)(spec_key[i] >> 32) * tb->n_b2 + (u32)spec_key[i]] = (i32)i;
        }
        t.spec_dense = spec_dense.empty() ? nullptr : spec_dense.data();
        t.pmask_words = (nP + 63) / 64;
        spec_p1.assign(tb->spec_p1_mask, tb->spec_p1_mask + (size_t)tb->n_specimens * t.pmask_words);
        spec_p2.assign(tb->spec_p2_mask, tb->spec_p2_mask + (size_t)tb->n_specimens * t.pmask_words);
        if (spec_p1.empty()) { spec_p1.push_back(0); spec_p2.push_back(0); }
        spec_pool.assign(tb->spec_pool, tb->spec_pool + tb->n_specimens);
        for (u32 i = 0; i < tb->n_specimens; ++i)
            if (tb->spec_pool[i] < -1 || tb->spec_pool[i] > 32767) return err("specimen pool id out of range");
        set_pointers(peq_rc.data(), peq_rcrev.data(), peq_fw.data(), b_len.data(), pb_barcode.data(),
                     pair_fwd.data(), pair_rev.data(), pair_pool.data(), spec_key.data(), spec_key_off.data(),
                     spec_row.data(), spec_p1.data(), spec_p2.data(), spec_pool.data());
        set_bword_pointers(bw_len.data(), bw_primer.data(), bw_row.data(), bw_valid.data(), bw_list.data(), beq.data());
        set_task_pointers(bt_g0.data(), bt_nw.data(), bt_row.data(), bt_eq.data());
        set_quad_pointers(bt_quad_row.data(), bt_quad.data());
        set_code_pointers(b_codes.data(), b_code_off.data(), bw_iupac.data());
        return true;
    }

    void set_bword_pointers(const unsigned char *len, const unsigned char *prim, const u32 *row, const u32 *valid,
                            const unsigned short *list, const u32 *eq) {
        t.bw_len = len; t.bw_primer = prim; t.bw_row = row; t.bw_valid = valid; t.bw_list = list; t.beq = eq;
    }

    // A/B switch (SMX_BARCODE_QUAD=1: narrow words of <= 8 barcodes take four work entries to a thread).  Off by
    // default: measured slower than the one-entry-per-thread task on config 2 (224 vs 197 us, profiles/r2_k_ab.md)
    static bool quad_enabled() { const char *e = getenv("SMX_BARCODE_QUAD"); return e && atoi(e) != 0; }
    void set_quad_pointers(const i32 *row, const u32 *quad) { t.bt_quad_row = row; t.bt_quad = quad; }

    void set_code_pointers(const unsigned char *codes, const u32 *off, const u32 *iupac) {
        t.b_codes = codes; t.b_code_off = off; t.bw_iupac = iupac;
    }

    void set_task_pointers(const unsigned short *g0, const unsigned char *nw, const u32 *row, const u32 *eq) {
        t.bt_g0 = g0; t.bt_nw = nw; t.bt_row = row; t.bt_eq = eq;
    }

    void set_pointers(const u64 *a, const u64 *b, const u64 *c, const unsigned char *e, const u32 *f,
                      const u32 *g, const u32 *h, const i32 *i, const u64 *j, const u32 *k, const u32 *l,
                      const u64 *m, const u64 *n, const i32 *o) {
        t.peq_rc = a; t.peq_rcrev = b; t.peq_fw = c; t.b_len = e; t.pb_barcode = f;
        t.pair_fwd = g; t.pair_rev = h; t.pair_pool = i; t.spec_key = j; t.spec_key_off = k; t.spec_row = l;
        t.spec_p1_mask = m; t.spec_p2_mask = n; t.spec_pool = o;
    }
};

}  // namespace smx
