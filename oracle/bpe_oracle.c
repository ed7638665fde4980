/*
 * bpe_oracle.c — CPU restatement of the byte-level BPE that BEAST trains and applies.
 *
 * TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's CPU legs,
 * never by the product package.
 *
 * The algorithm is NOT under /root/reference: the reference delegates it to the third-party Rust
 * library HF `tokenizers` (pinned tokenizers==0.21.4 in requirements.txt; 0.22.2 in this image):
 *   call sites  beast/beast_bpe_trainer.py:61-74  (ByteLevelBPETokenizer + BpeTrainer.train_from_iterator)
 *               beast/beast_bspline_bpe_tokenizer.py:197 (encode), :239 (decode)
 * This file restates the library's published algorithm (SURVEY.md Appendix A):
 *   A.1 string construction   chr(bin - min_token), initial alphabet chr(0..max-min)
 *   A.2 pre-tokenisation      ByteLevel(add_prefix_space=False, use_regex=True): the GPT-2 regex
 *   A.3 byte-level expansion  UTF-8 bytes -> GPT-2 bytes_to_unicode characters; ids by sorted codepoint
 *   A.4 training              exact arg-max pair count, ties -> smallest (id_a, id_b), min_frequency,
 *                             left-to-right non-overlapping merges, existing token strings re-used
 *   A.5 encode                per word: repeatedly merge the lowest-rank pair, leftmost first
 *   A.6 decode                ids -> byte-level characters -> bytes -> UTF-8 -> codepoints
 * Pinned against the live library (merges, vocabulary, ids) in tests/test_bpe_oracle.py and by the
 * golden files tests/golden/bpe_*.
 *
 * Shifted bins up to 0xD7FF (below the surrogates, which Python cannot hand to the library); the
 * character classes of codepoints >= 256 are supplied by the caller (bpe_oracle_set_classes: Unicode
 * general categories L*, N*, White_Space, as Oniguruma's \p{L} \p{N} \s).  vocab_size <= 8192.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define CLS_O 0
#define CLS_L 1
#define CLS_N 2
#define CLS_S 3

#define MAXCP 65536
static uint8_t g_cls[MAXCP];
static uint16_t g_b2u[256];     /* byte -> byte-level character (GPT-2 bytes_to_unicode) */
static int g_init = 0;

static void init_tables(void) {
    if (g_init) return;
    memset(g_cls, CLS_O, sizeof(g_cls));
    /* \s */
    const int ws[] = {9, 10, 11, 12, 13, 32, 133, 160};
    for (unsigned i = 0; i < sizeof(ws) / sizeof(ws[0]); ++i) g_cls[ws[i]] = CLS_S;
    /* \p{N} */
    for (int c = 48; c <= 57; ++c) g_cls[c] = CLS_N;
    const int nn[] = {178, 179, 185, 188, 189, 190};
    for (unsigned i = 0; i < sizeof(nn) / sizeof(nn[0]); ++i) g_cls[nn[i]] = CLS_N;
    /* \p{L} */
    for (int c = 65; c <= 90; ++c) g_cls[c] = CLS_L;
    for (int c = 97; c <= 122; ++c) g_cls[c] = CLS_L;
    g_cls[170] = g_cls[181] = g_cls[186] = CLS_L;
    for (int c = 192; c <= 214; ++c) g_cls[c] = CLS_L;
    for (int c = 216; c <= 246; ++c) g_cls[c] = CLS_L;
    for (int c = 248; c <= 255; ++c) g_cls[c] = CLS_L;
    /* bytes_to_unicode: printable bytes map to themselves, the other 68 to U+0100.. in byte order */
    int n = 0;
    for (int b = 0; b < 256; ++b) {
        int keep = (b >= 33 && b <= 126) || (b >= 161 && b <= 172) || (b >= 174 && b <= 255);
        g_b2u[b] = keep ? (uint16_t)b : (uint16_t)(256 + n++);
    }
    g_init = 1;
}

/* Classes of codepoints >= 256 (0 = other, 1 = letter, 2 = number, 3 = white space). */
void bpe_oracle_set_classes(const uint8_t* tab, int n) {
    init_tables();
    for (int c = 256; c < n && c < MAXCP; ++c) g_cls[c] = tab[c];
}

/* A.2: mark the first codepoint of every pre-token. */
static void pretokenize(const uint16_t* cp, int n, uint8_t* ws) {
    memset(ws, 0, (size_t)n);
    int i = 0;
    while (i < n) {
        ws[i] = 1;
        int c = cp[i];
        if (c == 39 && i + 1 < n) {                          /* 's|'t|'re|'ve|'m|'ll|'d */
            int d = cp[i + 1];
            if (d == 's' || d == 't' || d == 'm' || d == 'd') { i += 2; continue; }
            if (i + 2 < n) {
                int e = cp[i + 2];
                if ((d == 'r' && e == 'e') || (d == 'v' && e == 'e') || (d == 'l' && e == 'l')) { i += 3; continue; }
            }
        }
        int start = i;
        if (c == 32 && i + 1 < n && g_cls[cp[i + 1]] != CLS_S) start = i + 1;   /* " ?" prefix */
        int k = g_cls[cp[start]];
        if (k != CLS_S) {                                    /* ?\p{L}+ | ?\p{N}+ | ?[^\s\p{L}\p{N}]+ */
            int j = start + 1;
            while (j < n && g_cls[cp[j]] == k) ++j;
            i = j;
            continue;
        }
        int j = i + 1;                                       /* whitespace run [i, j) */
        while (j < n && g_cls[cp[j]] == CLS_S) ++j;
        if (j == n) { i = j; continue; }                     /* \s+(?!\S) at end of text */
        if (j - i >= 2) { i = j - 1; continue; }             /* \s+(?!\S): leave the last blank */
        i = j;                                               /* \s+ : a single non-space blank */
    }
}

/* A.3: codepoints -> bytes with word-start flags on the first byte of each pre-token. */
static int expand(const uint16_t* cp, const uint8_t* ws, int n, uint8_t* bytes, uint8_t* bws) {
    int m = 0;
    for (int i = 0; i < n; ++i) {
        int c = cp[i];
        if (c < 0x80) { bytes[m] = (uint8_t)c; bws[m++] = ws[i]; }
        else if (c < 0x800) {
            bytes[m] = (uint8_t)(0xC0 | (c >> 6)); bws[m++] = ws[i];
            bytes[m] = (uint8_t)(0x80 | (c & 0x3F)); bws[m++] = 0;
        } else {
            bytes[m] = (uint8_t)(0xE0 | (c >> 12)); bws[m++] = ws[i];
            bytes[m] = (uint8_t)(0x80 | ((c >> 6) & 0x3F)); bws[m++] = 0;
            bytes[m] = (uint8_t)(0x80 | (c & 0x3F)); bws[m++] = 0;
        }
    }
    return m;
}

/* ------------------------------------------------------------------ token table */
typedef struct {
    int n;              /* number of tokens */
    int cap_chars;
    int* off;           /* [n+1] offsets into chars */
    uint16_t* chars;    /* byte-level characters */
} tokens_t;

static int tok_len(const tokens_t* t, int id) { return t->off[id + 1] - t->off[id]; }

static int tok_find(const tokens_t* t, const uint16_t* s, int len) {
    for (int i = 0; i < t->n; ++i)
        if (tok_len(t, i) == len && memcmp(t->chars + t->off[i], s, (size_t)len * 2) == 0) return i;
    return -1;
}

/* ------------------------------------------------------------------ word dictionary (dedup with counts) */
typedef struct { int off, len; long long count; } word_t;

static uint64_t hash_bytes(const uint8_t* p, int n) {
    uint64_t h = 1469598103934665603ull;
    for (int i = 0; i < n; ++i) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}

/*
 * Train.  bins [n_seq, seq_len] int64.  Outputs (caller-allocated):
 *   vocab_off [vocab_size+1], vocab_chars [<= vocab_chars_cap]  byte-level characters of every token, id order
 *   merges [3 * vocab_size] : (id_a, id_b, id_new) in rank order
 * Returns 0 on success; *n_vocab_out, *n_merges_out set.  Negative on error.
 */
/*
 * bpe_oracle_train_ex adds what FIGBPE's other arguments reach in the library (beast/beast_bpe_trainer.py:46, 53, 76-98):
 *   row_off [n_seq+1] (nullable): sequences of unequal length, sequence s = bins[row_off[s] .. row_off[s+1])
 *   special tokens (n_special strings, UTF-16 code units in special_chars / special_off): BpeTrainer puts them
 *   into the vocabulary FIRST, in order, duplicates skipped; the alphabet follows, skipping characters that
 *   already are a (single-character) special token — such a character then carries the special token's id.
 */
int bpe_oracle_train_ex(const int64_t* bins, int64_t n_seq, int64_t seq_len, const int64_t* row_off, int64_t min_token,
                        int64_t max_token, int vocab_size, int min_frequency, int n_special, const int32_t* special_off,
                        const uint16_t* special_chars, int32_t* vocab_off, uint16_t* vocab_chars,
                        int64_t vocab_chars_cap, int32_t* merges, int32_t* n_vocab_out, int32_t* n_merges_out) {
    init_tables();
    if (max_token - min_token > 0xD7FF || max_token < min_token) return -2;
    if (vocab_size < 1 || vocab_size > 8192) return -2;
    if (max_token - min_token + 69 + n_special > 8192) return -2;          /* dense V x V counts */
    const int R = (int)(max_token - min_token);
    int L = (int)seq_len;
    if (row_off) {
        L = 1;
        for (int64_t s = 0; s < n_seq; ++s) if (row_off[s + 1] - row_off[s] > L) L = (int)(row_off[s + 1] - row_off[s]);
    }
    const int Lmax = L;

    /* pass 1: pre-tokenise, expand, collect unique words with counts */
    uint16_t* cp = (uint16_t*)malloc(((size_t)L + 1) * 2);
    uint8_t* ws = (uint8_t*)malloc((size_t)L + 1);
    uint8_t* by = (uint8_t*)malloc((size_t)3 * L + 3);
    uint8_t* bws = (uint8_t*)malloc((size_t)3 * L + 3);
    size_t pool_cap = 1 << 20, pool_n = 0;
    uint8_t* pool = (uint8_t*)malloc(pool_cap);
    size_t words_cap = 1 << 16, n_words = 0;
    word_t* words = (word_t*)malloc(words_cap * sizeof(word_t));
    size_t ht_cap = 1 << 18;
    int64_t* ht = (int64_t*)malloc(ht_cap * sizeof(int64_t));
    for (size_t i = 0; i < ht_cap; ++i) ht[i] = -1;
    uint8_t seen[256];
    memset(seen, 0, sizeof(seen));
    for (int64_t s = 0; s < n_seq; ++s) {
        const int64_t base = row_off ? row_off[s] : s * Lmax;
        L = row_off ? (int)(row_off[s + 1] - row_off[s]) : Lmax;
        for (int i = 0; i < L; ++i) {
            int64_t v = bins[base + i] - min_token;
            if (v < 0 || v > 0xD7FF) { free(cp); free(ws); free(by); free(bws); free(pool); free(words); free(ht); return -3; }
            cp[i] = (uint16_t)v;
        }
        pretokenize(cp, L, ws);
        int m = expand(cp, ws, L, by, bws);
        int i = 0;
        while (i < m) {
            int j = i + 1;
            while (j < m && !bws[j]) ++j;
            const int len = j - i;
            for (int q = i; q < j; ++q) seen[by[q]] = 1;
            uint64_t h = hash_bytes(by + i, len);
            size_t slot = h & (ht_cap - 1);
            for (;;) {
                int64_t w = ht[slot];
                if (w < 0) {
                    if (pool_n + (size_t)len > pool_cap) { pool_cap *= 2; pool = (uint8_t*)realloc(pool, pool_cap); }
                    if (n_words == words_cap) { words_cap *= 2; words = (word_t*)realloc(words, words_cap * sizeof(word_t)); }
                    memcpy(pool + pool_n, by + i, (size_t)len);
                    words[n_words].off = (int)pool_n; words[n_words].len = len; words[n_words].count = 1;
                    pool_n += (size_t)len;
                    ht[slot] = (int64_t)n_words++;
                    if (n_words * 2 > ht_cap) {              /* grow + rehash */
                        size_t nc = ht_cap * 4;
                        int64_t* nh = (int64_t*)malloc(nc * sizeof(int64_t));
                        for (size_t z = 0; z < nc; ++z) nh[z] = -1;
                        for (size_t z = 0; z < n_words; ++z) {
                            size_t sl = hash_bytes(pool + words[z].off, words[z].len) & (nc - 1);
                            while (nh[sl] >= 0) sl = (sl + 1) & (nc - 1);
                            nh[sl] = (int64_t)z;
                        }
                        free(ht); ht = nh; ht_cap = nc;
                    }
                    break;
                }
                if (words[w].len == len && memcmp(pool + words[w].off, by + i, (size_t)len) == 0) { words[w].count++; break; }
                slot = (slot + 1) & (ht_cap - 1);
            }
            i = j;
        }
    }
    free(cp); free(ws); free(by); free(bws); free(ht);

    /* alphabet: chr(0..R) U seen byte-level characters, ids by sorted codepoint (A.3) */
    uint8_t* in_alpha = (uint8_t*)calloc(MAXCP, 1);
    for (int c = 0; c <= R; ++c) in_alpha[c] = 1;
    for (int b = 0; b < 256; ++b) if (seen[b]) in_alpha[g_b2u[b]] = 1;
    tokens_t tk;
    tk.n = 0; tk.off = vocab_off; tk.chars = vocab_chars; tk.cap_chars = (int)vocab_chars_cap;
    int* char_to_id = (int*)malloc(sizeof(int) * MAXCP);
    tk.off[0] = 0;
    for (int i = 0; i < n_special; ++i) {                    /* special tokens first, duplicates skipped */
        const int len = special_off[i + 1] - special_off[i];
        if (tok_find(&tk, special_chars + special_off[i], len) >= 0) continue;
        memcpy(tk.chars + tk.off[tk.n], special_chars + special_off[i], (size_t)len * 2);
        tk.off[tk.n + 1] = tk.off[tk.n] + len;
        tk.n++;
    }
    for (int c = 0; c < MAXCP; ++c) {
        char_to_id[c] = -1;
        if (!in_alpha[c]) continue;
        const uint16_t cc = (uint16_t)c;
        const int have = tok_find(&tk, &cc, 1);              /* only a special token can already hold this string */
        if (have >= 0) { char_to_id[c] = have; continue; }
        char_to_id[c] = tk.n;                                /* the whole alphabet is kept even if it exceeds vocab_size */
        tk.chars[tk.off[tk.n]] = (uint16_t)c;
        tk.off[tk.n + 1] = tk.off[tk.n] + 1;
        tk.n++;
    }
    /* words as id arrays (in place over a new int pool) */
    int* sym = (int*)malloc((pool_n + 1) * sizeof(int));
    for (size_t w = 0; w < n_words; ++w)
        for (int q = 0; q < words[w].len; ++q) sym[words[w].off + q] = char_to_id[g_b2u[pool[words[w].off + q]]];
    free(pool); free(in_alpha); free(char_to_id);

    const int V = vocab_size > tk.n ? vocab_size : tk.n;     /* caller sizes vocab_off / merges for max(vocab_size, 512) */
    long long* cnt = (long long*)calloc((size_t)V * V, sizeof(long long));
    for (size_t w = 0; w < n_words; ++w) {
        const int* s = sym + words[w].off;
        for (int q = 0; q + 1 < words[w].len; ++q) cnt[(size_t)s[q] * V + s[q + 1]] += words[w].count;
    }
    int n_merges = 0;
    uint16_t* tmp = (uint16_t*)malloc(sizeof(uint16_t) * 70000);
    while (tk.n < vocab_size) {
        /* exact arg-max; ties -> smallest (a, b): first strictly-greater in flat order */
        long long best = 0; int ba = -1, bb = -1;
        const int cur = tk.n;
        for (int a = 0; a < cur; ++a) {
            const long long* row = cnt + (size_t)a * V;
            for (int b = 0; b < cur; ++b) if (row[b] > best) { best = row[b]; ba = a; bb = b; }
        }
        if (ba < 0 || best < 1 || best < min_frequency) break;
        /* new token string; an existing string keeps its id (the merge is still recorded) */
        int la = tok_len(&tk, ba), lb = tok_len(&tk, bb);
        if (la + lb > 60000) break;
        memcpy(tmp, tk.chars + tk.off[ba], (size_t)la * 2);
        memcpy(tmp + la, tk.chars + tk.off[bb], (size_t)lb * 2);
        int nid = tok_find(&tk, tmp, la + lb);
        if (nid < 0) {
            if (tk.off[tk.n] + la + lb > tk.cap_chars) { free(sym); free(words); free(cnt); free(tmp); return -4; }
            nid = tk.n;
            memcpy(tk.chars + tk.off[nid], tmp, (size_t)(la + lb) * 2);
            tk.off[nid + 1] = tk.off[nid] + la + lb;
            tk.n++;
        }
        merges[3 * n_merges] = ba; merges[3 * n_merges + 1] = bb; merges[3 * n_merges + 2] = nid;
        n_merges++;
        /* apply left to right, non-overlapping, in every word; recount the touched words */
        for (size_t w = 0; w < n_words; ++w) {
            int* s = sym + words[w].off;
            int len = words[w].len, hit = 0;
            for (int q = 0; q + 1 < len; ++q) if (s[q] == ba && s[q + 1] == bb) { hit = 1; break; }
            if (!hit) continue;
            for (int q = 0; q + 1 < len; ++q) cnt[(size_t)s[q] * V + s[q + 1]] -= words[w].count;
            int o = 0;
            for (int q = 0; q < len;) {
                if (q + 1 < len && s[q] == ba && s[q + 1] == bb) { s[o++] = nid; q += 2; }
                else s[o++] = s[q++];
            }
            words[w].len = len = o;
            for (int q = 0; q + 1 < len; ++q) cnt[(size_t)s[q] * V + s[q + 1]] += words[w].count;
        }
        if (n_merges >= vocab_size) break;
    }
    free(sym); free(words); free(cnt); free(tmp);
    *n_vocab_out = tk.n;
    *n_merges_out = n_merges;
    return 0;
}

int bpe_oracle_train(const int64_t* bins, int64_t n_seq, int64_t seq_len, int64_t min_token, int64_t max_token,
                     int vocab_size, int min_frequency, int32_t* vocab_off, uint16_t* vocab_chars,
                     int64_t vocab_chars_cap, int32_t* merges, int32_t* n_vocab_out, int32_t* n_merges_out) {
    return bpe_oracle_train_ex(bins, n_seq, seq_len, NULL, min_token, max_token, vocab_size, min_frequency, 0, NULL, NULL,
                               vocab_off, vocab_chars, vocab_chars_cap, merges, n_vocab_out, n_merges_out);
}

/* ------------------------------------------------------------------ encode / decode */
typedef struct {
    int n_vocab, n_merges, V;
    int* char_to_id;    /* [MAXCP] */
    int32_t* rank;      /* [V*V] merge rank or -1 */
    int32_t* newid;     /* [V*V] */
    int32_t* off;       /* [n_vocab+1] */
    uint16_t* chars;
} model_t;

void* bpe_oracle_model_new(const int32_t* vocab_off, const uint16_t* vocab_chars, int n_vocab, const int32_t* merges,
                           int n_merges) {
    init_tables();
    model_t* m = (model_t*)calloc(1, sizeof(model_t));
    m->n_vocab = n_vocab; m->n_merges = n_merges; m->V = n_vocab;
    m->off = (int32_t*)malloc(sizeof(int32_t) * (size_t)(n_vocab + 1));
    memcpy(m->off, vocab_off, sizeof(int32_t) * (size_t)(n_vocab + 1));
    m->chars = (uint16_t*)malloc(sizeof(uint16_t) * (size_t)(vocab_off[n_vocab] + 1));
    memcpy(m->chars, vocab_chars, sizeof(uint16_t) * (size_t)vocab_off[n_vocab]);
    m->char_to_id = (int*)malloc(sizeof(int) * MAXCP);
    for (int c = 0; c < MAXCP; ++c) m->char_to_id[c] = -1;
    for (int i = 0; i < n_vocab; ++i)
        if (vocab_off[i + 1] - vocab_off[i] == 1 && m->char_to_id[vocab_chars[vocab_off[i]]] < 0)
            m->char_to_id[vocab_chars[vocab_off[i]]] = i;
    m->rank = (int32_t*)malloc(sizeof(int32_t) * (size_t)m->V * m->V);
    m->newid = (int32_t*)malloc(sizeof(int32_t) * (size_t)m->V * m->V);
    for (size_t i = 0; i < (size_t)m->V * m->V; ++i) { m->rank[i] = -1; m->newid[i] = -1; }
    for (int r = 0; r < n_merges; ++r) {
        size_t key = (size_t)merges[3 * r] * m->V + merges[3 * r + 1];
        if (m->rank[key] < 0) { m->rank[key] = r; m->newid[key] = merges[3 * r + 2]; }
    }
    return m;
}

void bpe_oracle_model_free(void* p) {
    model_t* m = (model_t*)p;
    if (!m) return;
    free(m->rank); free(m->newid); free(m->off); free(m->chars); free(m->char_to_id); free(m);
}

/* Encode one sequence of shifted bins.  ids_out must hold 3*n entries.  Returns the id count. */
int bpe_oracle_encode(const void* p, const int64_t* shifted, int n, int32_t* ids_out) {
    const model_t* m = (const model_t*)p;
    uint16_t* cp = (uint16_t*)malloc(((size_t)n + 1) * 2);
    uint8_t* ws = (uint8_t*)malloc((size_t)n + 1);
    uint8_t* by = (uint8_t*)malloc((size_t)3 * n + 3);
    uint8_t* bws = (uint8_t*)malloc((size_t)3 * n + 3);
    int* w = (int*)malloc(sizeof(int) * ((size_t)3 * n + 3));
    for (int i = 0; i < n; ++i) cp[i] = (uint16_t)shifted[i];
    pretokenize(cp, n, ws);
    int mlen = expand(cp, ws, n, by, bws);
    int out = 0, i = 0;
    while (i < mlen) {
        int j = i + 1;
        while (j < mlen && !bws[j]) ++j;
        int len = 0;
        for (int q = i; q < j; ++q) {                        /* characters outside the vocabulary are dropped (no unk) */
            int id = m->char_to_id[g_b2u[by[q]]];
            if (id >= 0) w[len++] = id;
        }
        for (;;) {                                           /* lowest rank, leftmost first */
            int best = -1, bp = -1;
            for (int q = 0; q + 1 < len; ++q) {
                int r = m->rank[(size_t)w[q] * m->V + w[q + 1]];
                if (r >= 0 && (best < 0 || r < best)) { best = r; bp = q; }
            }
            if (best < 0) break;
            w[bp] = m->newid[(size_t)w[bp] * m->V + w[bp + 1]];
            memmove(w + bp + 1, w + bp + 2, sizeof(int) * (size_t)(len - bp - 2));
            --len;
        }
        for (int q = 0; q < len; ++q) ids_out[out++] = w[q];
        i = j;
    }
    free(cp); free(ws); free(by); free(bws); free(w);
    return out;
}

/* Encode n_seq rows of L shifted bins: the ids of row s land at ids_out[off_out[s] .. off_out[s + 1]).  ids_out holds
 * ids_cap entries (3 * n_seq * L always suffice).  Returns the total id count, or -1 if ids_cap is too small. */
int64_t bpe_oracle_encode_batch(const void* p, const int64_t* shifted, int64_t n_seq, int L, int32_t* ids_out,
                                int64_t ids_cap, int64_t* off_out) {
    int32_t* row = (int32_t*)malloc(sizeof(int32_t) * ((size_t)3 * L + 3));
    off_out[0] = 0;
    for (int64_t s = 0; s < n_seq; ++s) {
        const int n = bpe_oracle_encode(p, shifted + s * L, L, row);
        if (off_out[s] + n > ids_cap) { free(row); return -1; }
        memcpy(ids_out + off_out[s], row, sizeof(int32_t) * (size_t)n);
        off_out[s + 1] = off_out[s] + n;
    }
    free(row);
    return off_out[n_seq];
}

/* Decode ids -> codepoints (before adding min_token).  Returns the count, or -1 on an unknown id /
 * a byte-level character outside the 256-entry map, -2 on invalid UTF-8, -3 if out_cap is too small. */
int bpe_oracle_decode(const void* p, const int32_t* ids, int n, int64_t* out, int out_cap) {
    const model_t* m = (const model_t*)p;
    static int u2b[512];
    static int u2b_init = 0;
    if (!u2b_init) { for (int c = 0; c < 512; ++c) u2b[c] = -1; for (int b = 0; b < 256; ++b) u2b[g_b2u[b]] = b; u2b_init = 1; }
    int cnt = 0, pending = 0, acc = 0;
    for (int i = 0; i < n; ++i) {
        if (ids[i] < 0 || ids[i] >= m->n_vocab) return -1;
        for (int q = m->off[ids[i]]; q < m->off[ids[i] + 1]; ++q) {
            int ch = m->chars[q];
            int b = ch < 512 ? u2b[ch] : -1;
            if (b < 0) return -1;
            if (pending) {
                if ((b & 0xC0) != 0x80) return -2;
                acc = (acc << 6) | (b & 0x3F);
                if (--pending == 0) { if (cnt >= out_cap) return -3; out[cnt++] = acc; }
            } else if (b < 0x80) { if (cnt >= out_cap) return -3; out[cnt++] = b; }
            else if ((b & 0xE0) == 0xC0) { acc = b & 0x1F; pending = 1; }
            else if ((b & 0xF0) == 0xE0) { acc = b & 0x0F; pending = 2; }
            else if ((b & 0xF8) == 0xF0) { acc = b & 0x07; pending = 3; }
            else return -2;
        }
    }
    if (pending) return -2;
    return cnt;
}

/* Pre-tokeniser alone, for unit tests: ws_out[i] = 1 where a pre-token starts. */
void bpe_oracle_pretokenize(const uint16_t* cp, int n, uint8_t* ws_out) {
    init_tables();
    pretokenize(cp, n, ws_out);
}
