/*
 * transcript.c -- Keccak-f[1600], STROBE-128 subset, Merlin v1.0 transcripts and the ChaCha20 RNG for
 * the CPU oracle (test infrastructure, see eg_oracle.h).
 *
 * Replaces the un-vendored crates merlin 3.0.0 (+ keccak 0.1.6) and rand_chacha 0.10.0 / rand_core
 * as used by src/proofs/mod.rs:29-57, src/group/mod.rs:37-62 and tests/snapshots.rs:32.
 * Restated from: FIPS 202 (Keccak-f), STROBE v1.0.2 (strobe.sourceforge.io/specs), the Merlin
 * transcript framing (merlin.cool/transcript/ops.html), RFC 8439 2.3 (ChaCha20 block, here with a
 * 64-bit counter and zero nonce as rand_chacha does), PCG32 seed expansion (rand_core).
 */
#include "eg_oracle.h"
#include <string.h>

/* ---------------------------------------------------------------- Keccak-f[1600] */

static const uint64_t KECCAK_RC[24] = {
    0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL,
    0x000000000000808bULL, 0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL,
    0x000000000000008aULL, 0x0000000000000088ULL, 0x0000000080008009ULL, 0x000000008000000aULL,
    0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL, 0x8000000000008003ULL,
    0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,
    0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL};
static const int KECCAK_ROT[24] = {1, 3, 6, 10, 15, 21, 28, 36, 45, 55, 2, 14, 27, 41, 56, 8, 25, 43, 62, 18, 39, 61, 20, 44};
static const int KECCAK_PIL[24] = {10, 7, 11, 17, 18, 3, 5, 16, 8, 21, 24, 4, 15, 23, 19, 13, 12, 2, 20, 14, 22, 9, 6, 1};

#define ROL64(x, n) (((x) << (n)) | ((x) >> (64 - (n))))

void eo_keccak_f1600(uint8_t state[200]) {
    uint64_t a[25], bc[5], t;
    for (int i = 0; i < 25; i++) {
        a[i] = 0;
        for (int j = 0; j < 8; j++) a[i] |= (uint64_t)state[8 * i + j] << (8 * j);
    }
    for (int round = 0; round < 24; round++) {
        for (int i = 0; i < 5; i++) bc[i] = a[i] ^ a[i + 5] ^ a[i + 10] ^ a[i + 15] ^ a[i + 20];
        for (int i = 0; i < 5; i++) {
            t = bc[(i + 4) % 5] ^ ROL64(bc[(i + 1) % 5], 1);
            for (int j = 0; j < 25; j += 5) a[j + i] ^= t;
        }
        t = a[1];
        for (int i = 0; i < 24; i++) {
            int j = KECCAK_PIL[i];
            uint64_t b = a[j];
            a[j] = ROL64(t, KECCAK_ROT[i]);
            t = b;
        }
        for (int j = 0; j < 25; j += 5) {
            for (int i = 0; i < 5; i++) bc[i] = a[j + i];
            for (int i = 0; i < 5; i++) a[j + i] ^= (~bc[(i + 1) % 5]) & bc[(i + 2) % 5];
        }
        a[0] ^= KECCAK_RC[round];
    }
    for (int i = 0; i < 25; i++)
        for (int j = 0; j < 8; j++) state[8 * i + j] = (uint8_t)(a[i] >> (8 * j));
}

/* ---------------------------------------------------------------- STROBE-128 (subset used by Merlin) */

#define STROBE_R 166
#define FLAG_I 1
#define FLAG_A 2
#define FLAG_C 4
#define FLAG_T 8
#define FLAG_M 16
#define FLAG_K 32

static void strobe_run_f(eo_transcript *s) {
    s->state[s->pos] ^= s->pos_begin;
    s->state[s->pos + 1] ^= 0x04;
    s->state[STROBE_R + 1] ^= 0x80;
    eo_keccak_f1600(s->state);
    s->pos = 0;
    s->pos_begin = 0;
}

static void strobe_absorb(eo_transcript *s, const uint8_t *data, size_t len) {
    for (size_t i = 0; i < len; i++) {
        s->state[s->pos] ^= data[i];
        s->pos++;
        if (s->pos == STROBE_R) strobe_run_f(s);
    }
}

static void strobe_squeeze(eo_transcript *s, uint8_t *data, size_t len) {
    for (size_t i = 0; i < len; i++) {
        data[i] = s->state[s->pos];
        s->state[s->pos] = 0;
        s->pos++;
        if (s->pos == STROBE_R) strobe_run_f(s);
    }
}

static void strobe_begin_op(eo_transcript *s, uint8_t flags, int more) {
    if (more) return;   /* continuation of the previous operation (same flags) */
    uint8_t old_begin = s->pos_begin;
    s->pos_begin = s->pos + 1;
    s->cur_flags = flags;
    uint8_t hdr[2] = {old_begin, flags};
    strobe_absorb(s, hdr, 2);
    int force_f = (flags & (FLAG_C | FLAG_K)) != 0;
    if (force_f && s->pos != 0) strobe_run_f(s);
}

static void strobe_meta_ad(eo_transcript *s, const uint8_t *d, size_t n, int more) {
    strobe_begin_op(s, FLAG_M | FLAG_A, more);
    strobe_absorb(s, d, n);
}
static void strobe_ad(eo_transcript *s, const uint8_t *d, size_t n, int more) {
    strobe_begin_op(s, FLAG_A, more);
    strobe_absorb(s, d, n);
}
static void strobe_prf(eo_transcript *s, uint8_t *d, size_t n, int more) {
    strobe_begin_op(s, FLAG_I | FLAG_A | FLAG_C, more);
    strobe_squeeze(s, d, n);
}

static void strobe_new(eo_transcript *s, const char *protocol_label) {
    memset(s, 0, sizeof *s);
    const uint8_t hdr[6] = {1, STROBE_R + 2, 1, 0, 1, 96};
    memcpy(s->state, hdr, 6);
    memcpy(s->state + 6, "STROBEv1.0.2", 12);
    eo_keccak_f1600(s->state);
    s->pos = 0; s->pos_begin = 0; s->cur_flags = 0;
    strobe_meta_ad(s, (const uint8_t *)protocol_label, strlen(protocol_label), 0);
}

/* ---------------------------------------------------------------- Merlin */

static void le32(uint8_t b[4], uint32_t x) { for (int i = 0; i < 4; i++) b[i] = (uint8_t)(x >> (8 * i)); }

void eo_transcript_append_message(eo_transcript *t, const char *label, const uint8_t *msg, size_t len) {
    uint8_t l[4];
    le32(l, (uint32_t)len);
    strobe_meta_ad(t, (const uint8_t *)label, strlen(label), 0);
    strobe_meta_ad(t, l, 4, 1);
    strobe_ad(t, msg, len, 0);
}

void eo_transcript_new(eo_transcript *t, const char *label) {
    strobe_new(t, "Merlin v1.0");
    eo_transcript_append_message(t, "dom-sep", (const uint8_t *)label, strlen(label));
}

void eo_transcript_append_u64(eo_transcript *t, const char *label, uint64_t x) {
    uint8_t b[8];
    for (int i = 0; i < 8; i++) b[i] = (uint8_t)(x >> (8 * i));
    eo_transcript_append_message(t, label, b, 8);
}

void eo_transcript_challenge_bytes(eo_transcript *t, const char *label, uint8_t *out, size_t len) {
    uint8_t l[4];
    le32(l, (uint32_t)len);
    strobe_meta_ad(t, (const uint8_t *)label, strlen(label), 0);
    strobe_meta_ad(t, l, 4, 1);
    strobe_prf(t, out, len, 0);
}

/* proofs/mod.rs:40-42 */
void eo_transcript_start_proof(eo_transcript *t, const char *label) {
    eo_transcript_append_message(t, "dom-sep", (const uint8_t *)label, strlen(label));
}

/* proofs/mod.rs:48-52 */
void eo_transcript_append_element(eo_transcript *t, const char *label, const eo_pt *p) {
    uint8_t b[32];
    eo_pt_encode(b, p);
    eo_transcript_append_message(t, label, b, 32);
}

/* proofs/mod.rs:54-56 -> ristretto.rs:34-38 */
void eo_transcript_challenge_scalar(eo_transcript *t, const char *label, eo_sc *out) {
    uint8_t b[64];
    eo_transcript_challenge_bytes(t, label, b, 64);
    eo_sc_from_wide(out, b);
}

/* ---------------------------------------------------------------- ChaCha20 RNG */

#define ROL32(x, n) (((x) << (n)) | ((x) >> (32 - (n))))
#define QR(a, b, c, d) \
    a += b; d ^= a; d = ROL32(d, 16); c += d; b ^= c; b = ROL32(b, 12); \
    a += b; d ^= a; d = ROL32(d, 8);  c += d; b ^= c; b = ROL32(b, 7)

_Static_assert(sizeof(eo_rng) == 40, "eo_rng is allocated by callers at 40 bytes (key[32] + block)");
_Static_assert(sizeof(EO_RNG_REPLAY_TAG) - 1 == 16, "the replay tag fills replay.tag");

size_t eo_rng_size(void) { return sizeof(eo_rng); }

void eo_rng_from_seed(eo_rng *r, const uint8_t seed[32], uint64_t first_block) {
    memcpy(r->key, seed, 32);
    r->block = first_block;
}

void eo_rng_from_blocks(eo_rng *r, const uint8_t *blocks, uint64_t n_blocks) {
    memcpy(r->replay.tag, EO_RNG_REPLAY_TAG, 16);
    r->replay.blocks = blocks;
    r->replay.n_blocks = n_blocks;
    r->block = 0;
}

static int rng_is_replay(const eo_rng *r) { return memcmp(r->replay.tag, EO_RNG_REPLAY_TAG, 16) == 0; }

int eo_rng_overrun(const eo_rng *r) { return rng_is_replay(r) && r->block > r->replay.n_blocks; }

uint64_t eo_rng_blocks_left(const eo_rng *r) {
    return rng_is_replay(r) && r->block < r->replay.n_blocks ? r->replay.n_blocks - r->block : 0;
}

void eo_rng_seed_from_u64(eo_rng *r, uint64_t state) {
    /* rand_core::SeedableRng::seed_from_u64: PCG32 output words fill the seed */
    const uint64_t MUL = 6364136223846793005ULL, INC = 11634580027462260723ULL;
    uint8_t seed[32];
    for (int i = 0; i < 8; i++) {
        state = state * MUL + INC;
        uint32_t xorshifted = (uint32_t)(((state >> 18) ^ state) >> 27);
        uint32_t rot = (uint32_t)(state >> 59);
        uint32_t x = (xorshifted >> rot) | (xorshifted << ((32 - rot) & 31));
        for (int j = 0; j < 4; j++) seed[4 * i + j] = (uint8_t)(x >> (8 * j));
    }
    eo_rng_from_seed(r, seed, 0);
}

void eo_rng_block(eo_rng *r, uint8_t out[64]) {
    if (rng_is_replay(r)) {
        /* past the end: a 0xff block, and block > n_blocks from now on (eo_rng_overrun) */
        if (r->block < r->replay.n_blocks) memcpy(out, r->replay.blocks + 64 * r->block, 64);
        else memset(out, 0xff, 64);
        if (r->block <= r->replay.n_blocks) r->block++;
        return;
    }
    uint32_t s[16], x[16];
    s[0] = 0x61707865; s[1] = 0x3320646e; s[2] = 0x79622d32; s[3] = 0x6b206574;
    for (int i = 0; i < 8; i++)
        s[4 + i] = (uint32_t)r->key[4 * i] | ((uint32_t)r->key[4 * i + 1] << 8) |
                   ((uint32_t)r->key[4 * i + 2] << 16) | ((uint32_t)r->key[4 * i + 3] << 24);
    s[12] = (uint32_t)r->block; s[13] = (uint32_t)(r->block >> 32);
    s[14] = 0; s[15] = 0;
    memcpy(x, s, sizeof x);
    for (int i = 0; i < 10; i++) {
        QR(x[0], x[4], x[8], x[12]); QR(x[1], x[5], x[9], x[13]);
        QR(x[2], x[6], x[10], x[14]); QR(x[3], x[7], x[11], x[15]);
        QR(x[0], x[5], x[10], x[15]); QR(x[1], x[6], x[11], x[12]);
        QR(x[2], x[7], x[8], x[13]); QR(x[3], x[4], x[9], x[14]);
    }
    for (int i = 0; i < 16; i++) {
        uint32_t w = x[i] + s[i];
        for (int j = 0; j < 4; j++) out[4 * i + j] = (uint8_t)(w >> (8 * j));
    }
    r->block++;
}

void eo_rng_scalar(eo_rng *r, eo_sc *out) {
    uint8_t b[64];
    eo_rng_block(r, b);
    eo_sc_from_wide(out, b);
}
