/*
 * gc_oracle.c -- CPU ORACLE (test infrastructure, not the product; see gc_oracle.h).
 *
 * Literal plain-C restatement of the reference rules on a mailbox board.  It is written
 * independently of the CUDA kernels (no bitboards, no shared tables) so that agreement
 * between the two is evidence, not tautology.  Every function cites the reference lines
 * it follows: "lib.rs" = /root/reference/src/lib.rs, "v2.py" =
 * /root/reference/gym_chess/envs/chess_v2.py.
 */
#include "gc_oracle.h"

#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* piece ids, lib.rs:11-17 */
enum { EMPTY = 0, KING = 1, QUEEN = 2, ROOK = 3, BISHOP = 4, KNIGHT = 5, PAWN = 6 };

/* lib.rs:41-50 */
static const int8_t DEFAULT_BOARD[64] = {
    -3, -5, -4, -2, -1, -4, -5, -3, /**/ -6, -6, -6, -6, -6, -6, -6, -6,
    0,  0,  0,  0,  0,  0,  0,  0,  /**/ 0,  0,  0,  0,  0,  0,  0,  0,
    0,  0,  0,  0,  0,  0,  0,  0,  /**/ 0,  0,  0,  0,  0,  0,  0,  0,
    6,  6,  6,  6,  6,  6,  6,  6,  /**/ 3,  5,  4,  2,  1,  4,  5,  3,
};

const int8_t *gco_default_board(void) { return DEFAULT_BOARD; }

/* piece values, lib.rs:19-25 + PIECES table lib.rs:121-226 (value by |id|, king = 0) */
static int piece_value(int id) {
    switch (id < 0 ? -id : id) {
    case PAWN: return 1;
    case KNIGHT: return 3;
    case BISHOP: return 3;
    case ROOK: return 5;
    case QUEEN: return 10;
    default: return 0; /* king, empty */
    }
}

typedef struct {
    int8_t r0, c0, r1, c1;
} mv_t;

typedef struct {
    mv_t m[GCO_MAX_MOVES];
    int n;
} mvlist_t;

static void push(mvlist_t *l, int r0, int c0, int r1, int c1) {
    if (l->n < GCO_MAX_MOVES) {
        mv_t *m = &l->m[l->n++];
        m->r0 = (int8_t)r0, m->c0 = (int8_t)c0, m->r1 = (int8_t)r1, m->c1 = (int8_t)c1;
    }
}

/* ---- helper predicates, lib.rs:1179-1238 ---- */
static int on_board(int r, int c) { return !(r < 0 || r > 7 || c < 0 || c > 7); } /* lib.rs:1190 */
static int sq_empty(const gco_state *s, int r, int c) { return s->board[r * 8 + c] == 0; } /* 1194 */
static int color_of(int id) { return id > 0 ? GCO_WHITE : GCO_BLACK; }                    /* ID_TO_COLOR */
static int piece_from_player(const gco_state *s, int player, int r, int c) {              /* lib.rs:1201 */
    int id = s->board[r * 8 + c];
    if (id == 0) return 0;
    return color_of(id) == player;
}
static int king_from_player(const gco_state *s, int player, int r, int c) { /* lib.rs:1217 */
    int id = s->board[r * 8 + c];
    if (id != KING && id != -KING) return 0;
    return color_of(id) == player;
}

/* lib.rs:1063-1081: (add, stop) */
static void playable_move(const gco_state *s, int player, int r, int c, int *add, int *stop) {
    if (!on_board(r, c)) { *add = 0, *stop = 1; return; }
    if (sq_empty(s, r, c)) { *add = 1, *stop = 0; return; }
    if (piece_from_player(s, player, r, c)) { *add = 0, *stop = 1; return; }
    /* any piece of the other player, the king included (lib.rs:1074 precedes 1077) */
    *add = 1, *stop = 1;
}

/* lib.rs:1089-1104 */
static void attacking_move(const gco_state *s, int player, int r, int c, int *add, int *stop) {
    (void)player;
    if (!on_board(r, c)) { *add = 0, *stop = 1; return; }
    if (sq_empty(s, r, c)) { *add = 1, *stop = 0; return; }
    *add = 1, *stop = 1;
}

/* lib.rs:1113-1140 */
static int king_playable_move(const gco_state *s, int player, int r, int c, const uint8_t *attmap) {
    if (!on_board(r, c)) return 0;
    if (attmap[r * 8 + c]) return 0;
    if (sq_empty(s, r, c) || piece_from_player(s, -player, r, c)) return 1;
    return 0; /* own piece */
}

/* lib.rs:1147-1174 */
static int king_attacking_move(const gco_state *s, int player, int r, int c, const uint8_t *attmap) {
    (void)s, (void)player;
    if (!on_board(r, c)) return 0;
    if (attmap[r * 8 + c]) return 0;
    return 1; /* empty, own or other piece */
}

/* ---- piece generators, lib.rs:789-964 ---- */
static void king_moves(const gco_state *s, int player, int r, int c, const uint8_t *attmap, int attack, mvlist_t *l) {
    static const int steps[8][2] = {{1, 0}, {-1, 0}, {0, 1}, {0, -1}, {1, 1}, {1, -1}, {-1, 1}, {-1, -1}}; /* 797 */
    for (int k = 0; k < 8; k++) {
        int rr = r + steps[k][0], cc = c + steps[k][1];
        int add = attack ? king_attacking_move(s, player, rr, cc, attmap) : king_playable_move(s, player, rr, cc, attmap);
        if (add) push(l, r, c, rr, cc);
    }
}

/* lib.rs:853-887 */
static void iterativesteps(const gco_state *s, int player, int r, int c, int dr, int dc, int attack, mvlist_t *l) {
    for (int k = 1;; k++) {
        int rr = r + k * dr, cc = c + k * dc, add, stop;
        if (attack) attacking_move(s, player, rr, cc, &add, &stop);
        else playable_move(s, player, rr, cc, &add, &stop);
        if (add) push(l, r, c, rr, cc);
        if (stop) break;
    }
}

static void rook_moves(const gco_state *s, int player, int r, int c, int attack, mvlist_t *l) {
    static const int steps[4][2] = {{-1, 0}, {1, 0}, {0, -1}, {0, 1}}; /* lib.rs:835 */
    for (int k = 0; k < 4; k++) iterativesteps(s, player, r, c, steps[k][0], steps[k][1], attack, l);
}

static void bishop_moves(const gco_state *s, int player, int r, int c, int attack, mvlist_t *l) {
    static const int steps[4][2] = {{-1, -1}, {-1, 1}, {1, -1}, {1, 1}}; /* lib.rs:845 */
    for (int k = 0; k < 4; k++) iterativesteps(s, player, r, c, steps[k][0], steps[k][1], attack, l);
}

static void queen_moves(const gco_state *s, int player, int r, int c, int attack, mvlist_t *l) { /* lib.rs:824 */
    rook_moves(s, player, r, c, attack, l);
    bishop_moves(s, player, r, c, attack, l);
}

static void knight_moves(const gco_state *s, int player, int r, int c, int attack, mvlist_t *l) {
    static const int steps[8][2] = {{-2, -1}, {-2, 1}, {2, -1}, {2, 1}, {-1, -2}, {-1, 2}, {1, -2}, {1, 2}}; /* 891 */
    for (int k = 0; k < 8; k++) {
        int rr = r + steps[k][0], cc = c + steps[k][1], add, stop;
        if (attack) attacking_move(s, player, rr, cc, &add, &stop);
        else playable_move(s, player, rr, cc, &add, &stop);
        if (add) push(l, r, c, rr, cc);
    }
}

/* lib.rs:918-964 */
static void pawn_moves(const gco_state *s, int player, int r, int c, int attack, mvlist_t *l) {
    int p = player; /* player.to_int() */
    int att[2][2] = {{r - p, c + 1}, {r - p, c - 1}};
    int r1 = r - p, r2 = r - 2 * p;
    if (attack) {
        for (int k = 0; k < 2; k++)
            if (on_board(att[k][0], att[k][1]) && !king_from_player(s, player, att[k][0], att[k][1]))
                push(l, r, c, att[k][0], att[k][1]);
    } else {
        if (on_board(r1, c) && s->board[r1 * 8 + c] == 0) push(l, r, c, r1, c);
        if (on_board(r2, c)) {
            if ((player == GCO_WHITE && r == 6) || (player == GCO_BLACK && r == 1)) {
                if (s->board[r2 * 8 + c] == 0) push(l, r, c, r2, c); /* jumped square not tested, lib.rs:942-954 */
            }
        }
        for (int k = 0; k < 2; k++)
            if (on_board(att[k][0], att[k][1]) && piece_from_player(s, -player, att[k][0], att[k][1]))
                push(l, r, c, att[k][0], att[k][1]);
    }
}

static void apply_move(const gco_state *s, int player, int is_castle, mv_t m, int castle, gco_state *out, int *reward,
                       int *err);
static void attack_map(const gco_state *s, int player, uint8_t *map);

/* lib.rs:634-667.  NOTE the `break` leaves only the inner loop: the king found in the LAST row
 * holding one wins (first column within that row). */
static int king_is_checked_map(const gco_state *s, int player, const uint8_t *attmap) {
    int king_id = KING * player, found = 0, kr = 0, kc = 0;
    for (int i = 0; i < 8; i++)
        for (int j = 0; j < 8; j++)
            if (s->board[i * 8 + j] == king_id) {
                found = 1, kr = i, kc = j;
                break;
            }
    if (!found) return 0;
    return attmap[kr * 8 + kc] != 0;
}

/* lib.rs:628-632 */
static int king_is_checked(const gco_state *s, int player) {
    uint8_t map[64];
    attack_map(s, -player, map);
    return king_is_checked_map(s, player, map);
}

/* lib.rs:612-626 */
static int move_leaves_king_checked(const gco_state *s, int player, mv_t m) {
    int from = s->board[m.r0 * 8 + m.c0];
    if ((player == GCO_WHITE && from == KING) || (player == GCO_BLACK && from == -KING)) return 0;
    gco_state nxt;
    int rew, err;
    apply_move(s, player, 0, m, 0, &nxt, &rew, &err);
    return king_is_checked(&nxt, player);
}

/* lib.rs:501-563 */
static void gen_possible_moves(const gco_state *s, int player, int attack, const uint8_t *attmap, mvlist_t *l) {
    l->n = 0;
    for (int i = 0; i < 8; i++)
        for (int j = 0; j < 8; j++) {
            int id = s->board[i * 8 + j];
            if (id == 0) continue;
            if (color_of(id) != player) continue;
            switch (id < 0 ? -id : id) {
            case KING: king_moves(s, player, i, j, attmap, attack, l); break;
            case QUEEN: queen_moves(s, player, i, j, attack, l); break;
            case ROOK: rook_moves(s, player, i, j, attack, l); break;
            case BISHOP: bishop_moves(s, player, i, j, attack, l); break;
            case KNIGHT: knight_moves(s, player, i, j, attack, l); break;
            case PAWN: pawn_moves(s, player, i, j, attack, l); break;
            default: break;
            }
        }
    if (attack) return;
    int w = 0; /* retain(), lib.rs:561 */
    for (int k = 0; k < l->n; k++)
        if (!move_leaves_king_checked(s, player, l->m[k])) l->m[w++] = l->m[k];
    l->n = w;
}

/* lib.rs:669-677 */
static void attack_map(const gco_state *s, int player, uint8_t *map) {
    uint8_t empty[64]; /* the attack-mode pass receives an EMPTY map, lib.rs:670-671 */
    mvlist_t l;        /* 8 KB; recursion depth is 2 (filter -> attack map) */
    memset(empty, 0, 64);
    memset(map, 0, 64);
    gen_possible_moves(s, player, 1, empty, &l);
    for (int k = 0; k < l.n; k++) map[l.m[k].r1 * 8 + l.m[k].c1] = 1;
}

/* lib.rs:966-1056.  The black branch compares with +ROOK/+KING exactly like the reference. */
static int calc_castle_moves(const gco_state *s, int player, const uint8_t *map, uint16_t *out) {
    int n = 0;
    const int8_t *b = s->board;
    if (player == GCO_WHITE) {
        if (b[7 * 8 + 0] == ROOK && b[7 * 8 + 1] == EMPTY && b[7 * 8 + 2] == EMPTY && b[7 * 8 + 3] == EMPTY &&
            b[7 * 8 + 4] == KING && !map[7 * 8 + 4] && !map[7 * 8 + 3] && !map[7 * 8 + 2])
            out[n++] = GCO_ACT_CASTLE_QS_WHITE;
        if (b[7 * 8 + 7] == ROOK && b[7 * 8 + 6] == EMPTY && b[7 * 8 + 5] == EMPTY && b[7 * 8 + 4] == KING &&
            !map[7 * 8 + 4] && !map[7 * 8 + 5] && !map[7 * 8 + 6])
            out[n++] = GCO_ACT_CASTLE_KS_WHITE;
    } else {
        if (b[0] == ROOK && b[1] == EMPTY && b[2] == EMPTY && b[3] == EMPTY && b[4] == KING && !map[4] && !map[3] &&
            !map[2])
            out[n++] = GCO_ACT_CASTLE_QS_BLACK;
        if (b[7] == ROOK && b[6] == EMPTY && b[5] == EMPTY && b[4] == KING && !map[4] && !map[5] && !map[6])
            out[n++] = GCO_ACT_CASTLE_KS_BLACK;
    }
    return n;
}

/* lib.rs:578-610 */
static int gen_castle_moves(const gco_state *s, int player, int attack, const uint8_t *map, uint16_t *out) {
    if (attack) return 0;
    if ((player == GCO_WHITE && !s->white_king_on_board) || (player == GCO_BLACK && !s->black_king_on_board)) return 0;
    if ((player == GCO_WHITE && (s->wk || s->wq)) || (player == GCO_BLACK && (s->bk || s->bq)))
        return calc_castle_moves(s, player, map, out);
    return 0;
}

/* lib.rs:679-784 (next_state): apply a normal move or a castle */
static void apply_move(const gco_state *s, int player, int is_castle, mv_t m, int castle, gco_state *out, int *reward,
                       int *err) {
    *out = *s;
    *reward = 0;
    *err = 0;
    int8_t *b = out->board;
    if (!is_castle) {
        int from = m.r0 * 8 + m.c0, to = m.r1 * 8 + m.c1;
        int piece = b[from], captured = b[to];
        if (piece == 0) { *err = -1; return; } /* panic!("Bad move - piece is empty !") */
        b[from] = 0;
        b[to] = (int8_t)piece;
        *reward += piece_value(captured);
        /* "Pawn becomes Queen": rows are the WRONG ends (lib.rs:703-704), kept as is */
        if (piece == PAWN || piece == -PAWN) {
            if ((player == GCO_WHITE && m.r1 == 7) || (player == GCO_BLACK && m.r1 == 0)) {
                b[to] = (int8_t)(QUEEN * player);
                *reward += 10;
            }
        }
        /* castling rights: only WHITE ids match (lib.rs:712, 720) */
        if (piece == KING) {
            if (player == GCO_WHITE) out->wk = 0, out->wq = 0;
            else out->bk = 0, out->bq = 0;
        } else if (piece == ROOK) {
            if (m.c0 == 0) {
                if (player == GCO_WHITE) out->wq = 0;
                else out->bq = 0;
            } else if (m.c0 == 7) {
                if (player == GCO_WHITE) out->wk = 0;
                else out->bk = 0;
            }
        }
    } else {
        switch (castle) {
        case GCO_ACT_CASTLE_KS_WHITE:
            b[60] = 0, b[61] = ROOK, b[62] = KING, b[63] = 0;
            out->wk = 0, out->wq = 0;
            break;
        case GCO_ACT_CASTLE_QS_WHITE:
            b[56] = 0, b[57] = 0, b[58] = KING, b[59] = ROOK, b[60] = 0;
            out->wk = 0, out->wq = 0;
            break;
        case GCO_ACT_CASTLE_KS_BLACK:
            b[4] = 0, b[5] = -ROOK, b[6] = -KING, b[7] = 0;
            out->bk = 0, out->bq = 0;
            break;
        case GCO_ACT_CASTLE_QS_BLACK:
            b[0] = 0, b[1] = 0, b[2] = -KING, b[3] = -ROOK, b[4] = 0;
            out->bk = 0, out->bq = 0;
            break;
        default: *err = -2; return;
        }
    }
    out->current_player = (int8_t)(-player); /* lib.rs:779-780 */
}

/* ------------------------------------------------------------------ engine level */

static int piece_is_on_board(const int8_t *b, int id) { /* lib.rs:1375 */
    for (int i = 0; i < 64; i++)
        if (b[i] == id) return 1;
    return 0;
}

void gco_state_new(gco_state *s, const int8_t *board, int player, int wk, int wq, int bk, int bq) {
    memcpy(s->board, board, 64);
    s->current_player = (int8_t)(player == GCO_BLACK ? GCO_BLACK : GCO_WHITE);
    s->white_king_on_board = (uint8_t)piece_is_on_board(board, KING);
    s->black_king_on_board = (uint8_t)piece_is_on_board(board, -KING);
    s->wk = (uint8_t)(wk != 0), s->wq = (uint8_t)(wq != 0), s->bk = (uint8_t)(bk != 0), s->bq = (uint8_t)(bq != 0);
    if (!s->white_king_on_board) s->wk = 0, s->wq = 0; /* lib.rs:315-318 */
    if (!s->black_king_on_board) s->bk = 0, s->bq = 0; /* lib.rs:319-322 */
    s->wchk = 0, s->bchk = 0;
}

static uint16_t mv_to_action(mv_t m) { return (uint16_t)((m.r0 * 8 + m.c0) * 64 + (m.r1 * 8 + m.c1)); }

/* lib.rs:460-486 + 1455-1480 */
int gco_get_possible_moves(const gco_state *s, int player, int attack, uint16_t *out, int cap) {
    uint8_t map[64];
    memset(map, 0, 64);
    if (!attack) attack_map(s, -player, map);
    mvlist_t l;
    gen_possible_moves(s, player, attack, map, &l);
    int n = 0;
    for (int k = 0; k < l.n && n < cap; k++) out[n++] = mv_to_action(l.m[k]);
    uint16_t c[2];
    int nc = gen_castle_moves(s, player, attack, map, c);
    for (int k = 0; k < nc && n < cap; k++) out[n++] = c[k];
    return n;
}

/* lib.rs:566-575 + 1482-1500 */
int gco_get_castle_moves(const gco_state *s, int player, uint16_t *out, int cap) {
    uint8_t map[64];
    attack_map(s, -player, map);
    uint16_t c[2];
    int nc = gen_castle_moves(s, player, 0, map, c), n = 0;
    for (int k = 0; k < nc && n < cap; k++) out[n++] = c[k];
    return n;
}

/* lib.rs:1386-1393 */
void gco_update_state(gco_state *s) {
    uint8_t map[64];
    attack_map(s, GCO_BLACK, map);
    s->wchk = (uint8_t)king_is_checked_map(s, GCO_WHITE, map);
    attack_map(s, GCO_WHITE, map);
    s->bchk = (uint8_t)king_is_checked_map(s, GCO_BLACK, map);
}

/* lib.rs:1422-1452 */
int gco_next_state(const gco_state *s, int player, int action, gco_state *out, int *reward, int *both_checked) {
    mv_t m = {0, 0, 0, 0};
    int is_castle = 0, err;
    if (action >= 4096 && action <= 4099) is_castle = 1;
    else if (action >= 0 && action < 4096) {
        int from = action / 64, to = action % 64;
        m.r0 = (int8_t)(from / 8), m.c0 = (int8_t)(from % 8), m.r1 = (int8_t)(to / 8), m.c1 = (int8_t)(to % 8);
    } else return -2;
    apply_move(s, player, is_castle, m, action, out, reward, &err);
    if (err) return err;
    gco_update_state(out);
    if (both_checked) *both_checked = out->wchk && out->bchk;
    return 0;
}

/* ------------------------------------------------------------------ Philox4x32-10 */

void gco_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0, c1 = n1, c2 = n2, c3 = n3;
        k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
    }
    out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}

uint32_t gco_draw_u32(uint64_t seed, uint32_t env_id, uint32_t episode, uint32_t step, uint32_t purpose) {
    uint32_t ctr[4] = {env_id, episode, step, purpose}, key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)}, o[4];
    gco_philox4x32_10(ctr, key, o);
    return o[0];
}

/* ------------------------------------------------------------------ env level (v2.py) */

static void env_movegen(gco_env *e, int player) { /* v2.py:573-582 (engine entry masks flags again) */
    gco_state tmp;
    gco_state_new(&tmp, e->st.board, e->st.current_player, e->st.wk, e->st.wq, e->st.bk, e->st.bq);
    e->n_legal = gco_get_possible_moves(&tmp, player, 0, e->legal, GCO_MAX_MOVES);
}

void gco_env_init(gco_env *e, const int8_t *initial_board, int agent_black, int opponent, uint64_t seed,
                  uint32_t env_id) {
    memset(e, 0, sizeof(*e));
    memcpy(e->initial_board, initial_board ? initial_board : DEFAULT_BOARD, 64);
    e->agent_black = agent_black, e->opponent = opponent, e->moves_max = 149;
    e->seed = seed, e->env_id = env_id, e->episode = 0;
    e->forced_bot_action = -1;
    e->hist_cap = 1024;
    e->hist = (int8_t *)malloc((size_t)e->hist_cap * 64);
    gco_env_reset(e);
}

void gco_env_free(gco_env *e) {
    free(e->hist);
    e->hist = NULL;
}

/* player_move, v2.py:393-412: returns reward, sets *rep when the pre-move board is seen a 3rd time */
static int env_player_move(gco_env *e, int action, int *reward, int *rep) {
    gco_state in, out;
    int both;
    /* engine entry: convert_py_state -> State::new masks the flags by the INPUT board (Q21) */
    gco_state_new(&in, e->st.board, e->st.current_player, e->st.wk, e->st.wq, e->st.bk, e->st.bq);
    int rc = gco_next_state(&in, e->st.current_player, action, &out, reward, &both);
    if (rc) return rc;
    /* encode_board() of the PRE-move board, v2.py:404-407 */
    int count = 1;
    for (int i = 0; i < e->hist_n; i++)
        if (memcmp(e->hist + (size_t)i * 64, e->st.board, 64) == 0) count++;
    if (e->hist_n == e->hist_cap) {
        e->hist_cap *= 2;
        e->hist = (int8_t *)realloc(e->hist, (size_t)e->hist_cap * 64);
    }
    memcpy(e->hist + (size_t)e->hist_n * 64, e->st.board, 64);
    e->hist_n++;
    *rep = count >= 3;
    /* state setter, v2.py:315-323: board + 4 castle flags + 2 check flags; current_player untouched */
    int8_t cur = e->st.current_player;
    e->st = out;
    e->st.current_player = cur;
    return 0;
}

/* v2.py:183-217 */
void gco_env_reset(gco_env *e) {
    e->done = 0;
    e->hist_n = 0;
    e->move_count = 0;
    e->wedged_bot = 0;
    e->step_in_episode = 0;
    e->last_bot_action = -1;
    gco_state_new(&e->st, e->initial_board, GCO_WHITE, 1, 1, 1, 1);
    gco_update_state(&e->st); /* engine.update_state(self.state): masked flags + check flags */
    env_movegen(e, GCO_WHITE);
    if (e->agent_black) {
        /* white opening ply by the opponent policy, v2.py:208-216 */
        uint32_t u = gco_draw_u32(e->seed, e->env_id, e->episode, 0, GCO_PURPOSE_RESET);
        if (e->n_legal > 0) {
            int a = e->legal[(uint32_t)(((uint64_t)u * (uint32_t)e->n_legal) >> 32)], r, rep;
            if (e->forced_bot_action >= 0) a = e->forced_bot_action;
            env_player_move(e, a, &r, &rep);
            e->last_bot_action = a;
        } else {
            e->wedged_bot = 1; /* reference: "resign" -> TypeError */
        }
        e->move_count += 1;
        e->st.current_player = GCO_BLACK;
        env_movegen(e, GCO_BLACK);
    }
}

int gco_env_pick(const gco_env *e, uint32_t u32) {
    if (e->n_legal <= 0) return GCO_ACT_RESIGN;
    return e->legal[(uint32_t)(((uint64_t)u32 * (uint32_t)e->n_legal) >> 32)];
}

static int king_checked_flag(const gco_env *e, int player) { return player == GCO_WHITE ? e->st.wchk : e->st.bchk; }

/* v2.py:219-294 */
int gco_env_step(gco_env *e, int action, int *reward, int *done) {
    uint32_t step_idx = e->step_in_episode++;
    e->last_bot_action = -1;
    /* action not in possible_actions -> (-10, self.done), checked BEFORE done (v2.py:240-242) */
    int valid = 0;
    for (int i = 0; i < e->n_legal; i++)
        if (e->legal[i] == action) { valid = 1; break; }
    if (!valid) { *reward = -10, *done = e->done; return 0; }
    if (e->done) { *reward = 0, *done = 1; return 0; }                       /* v2.py:245-251 */
    if (e->move_count > e->moves_max) { *reward = 0, *done = 1; return 0; } /* v2.py:252-258, done not latched */

    int R = -10, r, rep; /* v2.py:261 (sic) */
    env_player_move(e, action, &r, &rep);
    e->done = rep;
    R += r;
    e->st.current_player = (int8_t)(-e->st.current_player); /* switch_player, v2.py:267 */
    env_movegen(e, e->st.current_player);
    if (e->n_legal == 0 && king_checked_flag(e, e->st.current_player)) { e->done = 1, R += 100; } /* v2.py:270-272 */
    if (e->done) { *reward = R, *done = 1; return 0; }

    if (e->opponent == GCO_OPP_RANDOM) { /* v2.py:277-288 */
        if (e->n_legal == 0) {
            /* policy returns "resign" -> move_to_action -> None -> TypeError (Q9) */
            e->wedged_bot = 1;
            *reward = R, *done = 0;
            return 1;
        }
        uint32_t u = gco_draw_u32(e->seed, e->env_id, e->episode, step_idx, GCO_PURPOSE_BOT);
        int a = e->legal[(uint32_t)(((uint64_t)u * (uint32_t)e->n_legal) >> 32)];
        if (e->forced_bot_action >= 0) a = e->forced_bot_action; /* replay of a recorded bot move (tests) */
        e->last_bot_action = a;
        env_player_move(e, a, &r, &rep);
        e->done = rep;
        e->st.current_player = (int8_t)(-e->st.current_player);
        env_movegen(e, e->st.current_player);
        R -= r;
        if (e->n_legal == 0 && king_checked_flag(e, e->st.current_player)) { e->done = 1, R += -100; }
    }
    if (e->st.current_player == GCO_WHITE) e->move_count += 1; /* v2.py:291-292 */
    *reward = R, *done = e->done;
    return 0;
}

/* ------------------------------------------------------------------ bulk self-play drivers */

static void stats_add(gco_stats *a, const gco_stats *b) {
    a->steps += b->steps, a->plies += b->plies, a->episodes += b->episodes, a->mates += b->mates;
    a->repetitions += b->repetitions, a->caps += b->caps, a->wedged += b->wedged, a->invalid += b->invalid;
    a->reward_sum += b->reward_sum, a->legal_sum += b->legal_sum, a->in_check += b->in_check;
}

/* One sampled step with the same bookkeeping as the CUDA env's sampled step (DESIGN.md "sampled step"). */
void gco_selfplay(gco_env *e, uint64_t nsteps, gco_stats *st) {
    for (uint64_t t = 0; t < nsteps; t++) {
        uint32_t u = gco_draw_u32(e->seed, e->env_id, e->episode, e->step_in_episode, GCO_PURPOSE_AGENT);
        int a = gco_env_pick(e, u), r, d;
        int n_before = e->n_legal, was_done = e->done, capped = e->move_count > e->moves_max;
        st->legal_sum += (uint64_t)n_before;
        st->in_check += (uint64_t)king_checked_flag(e, e->st.current_player);
        int hist_before = e->hist_n;
        int raised = gco_env_step(e, a, &r, &d);
        st->steps++;
        st->plies += (uint64_t)(e->hist_n - hist_before);
        st->reward_sum += r;
        (void)raised;
        if (n_before == 0) st->invalid++;
        else if (was_done) {
        } else if (capped) st->caps++;
        else if (d) {
            if (e->n_legal == 0 && king_checked_flag(e, e->st.current_player)) st->mates++;
            else st->repetitions++;
        } else if (e->n_legal == 0) st->wedged++;
        int terminal = d || e->n_legal == 0;
        if (terminal) {
            st->episodes++;
            e->episode++;
            gco_env_reset(e);
        }
    }
}

/* Positions for the fixed movegen test set (tests/positions_1m.py): env `id` plays `nsteps` sampled self-play steps (same
 * draws and auto-reset as gco_selfplay) and the position BEFORE step t is recorded whenever t % every == id % every, so
 * every ply index of a game is equally likely.  Returns the number of positions written (<= cap). */
int gco_harvest(uint64_t seed, uint32_t env_lo, uint32_t env_hi, uint64_t nsteps, int every, int8_t *boards,
                int8_t *players, uint8_t *rights, int cap) {
    int n = 0;
    gco_stats st;
    memset(&st, 0, sizeof(st));
    for (uint32_t id = env_lo; id < env_hi && n < cap; id++) {
        gco_env e;
        gco_env_init(&e, NULL, 0, GCO_OPP_NONE, seed, id);
        for (uint64_t t = 0; t < nsteps && n < cap; t++) {
            if ((int)(t % (uint64_t)every) == (int)(id % (uint32_t)every)) {
                memcpy(boards + (size_t)n * 64, e.st.board, 64);
                players[n] = e.st.current_player;
                rights[(size_t)n * 4 + 0] = e.st.wk, rights[(size_t)n * 4 + 1] = e.st.wq;
                rights[(size_t)n * 4 + 2] = e.st.bk, rights[(size_t)n * 4 + 3] = e.st.bq;
                n++;
            }
            gco_selfplay(&e, 1, &st);
        }
        gco_env_free(&e);
    }
    return n;
}

typedef struct {
    uint64_t seed, nsteps;
    uint32_t lo, hi;
    gco_stats st;
} mt_arg;

static void *mt_worker(void *p) {
    mt_arg *a = (mt_arg *)p;
    memset(&a->st, 0, sizeof(a->st));
    for (uint32_t id = a->lo; id < a->hi; id++) {
        gco_env e;
        gco_env_init(&e, NULL, 0, GCO_OPP_NONE, a->seed, id);
        gco_selfplay(&e, a->nsteps, &a->st);
        gco_env_free(&e);
    }
    return NULL;
}

void gco_selfplay_mt(uint64_t seed, uint32_t env_lo, uint32_t env_hi, uint64_t nsteps_per_env, int threads,
                     gco_stats *st) {
    if (threads < 1) threads = 1;
    uint32_t n = env_hi - env_lo;
    if ((uint32_t)threads > n) threads = (int)(n ? n : 1);
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
    mt_arg *args = (mt_arg *)malloc(sizeof(mt_arg) * (size_t)threads);
    for (int t = 0; t < threads; t++) {
        args[t].seed = seed, args[t].nsteps = nsteps_per_env;
        args[t].lo = env_lo + (uint32_t)((uint64_t)n * (uint64_t)t / (uint64_t)threads);
        args[t].hi = env_lo + (uint32_t)((uint64_t)n * (uint64_t)(t + 1) / (uint64_t)threads);
        pthread_create(&th[t], NULL, mt_worker, &args[t]);
    }
    memset(st, 0, sizeof(*st));
    for (int t = 0; t < threads; t++) {
        pthread_join(th[t], NULL);
        stats_add(st, &args[t].st);
    }
    free(th);
    free(args);
}

/* ---- a persistent pool of envs: burn-in once, then timed steps on the same envs, so that the CPU arm of bench.py
 * (--impl reference) measures the same steady-state mix of game phases as the GPU arm; configured like the CUDA env
 * (opponent, agent colour, moves_max, template boards), it is also the reference of whole device batches */
struct gco_pool {
    gco_env *envs;
    uint32_t n;
};

typedef struct {
    gco_pool *pool;
    uint32_t lo, hi;
    uint64_t nsteps;
    uint32_t stagger; /* > 0: env i runs (i % stagger) steps more (spreads the episode phases of a pool) */
    gco_stats st;
} pool_arg;

static void *pool_worker(void *p) {
    pool_arg *a = (pool_arg *)p;
    memset(&a->st, 0, sizeof(a->st));
    for (uint32_t i = a->lo; i < a->hi; i++)
        gco_selfplay(&a->pool->envs[i], a->nsteps + (a->stagger ? (uint64_t)(i % a->stagger) : 0), &a->st);
    return NULL;
}

gco_pool *gco_pool_new_cfg(uint64_t seed, uint32_t env_lo, uint32_t env_hi, int opponent, int agent_black, int moves_max,
                           int n_templates, const int8_t *templates) {
    gco_pool *p = (gco_pool *)malloc(sizeof(gco_pool));
    p->n = env_hi - env_lo;
    p->envs = (gco_env *)malloc(sizeof(gco_env) * (size_t)p->n);
    for (uint32_t i = 0; i < p->n; i++) {
        const uint32_t id = env_lo + i; /* the device's template rule: global env id % n_templates */
        const int8_t *board = (templates && n_templates > 0) ? templates + (size_t)(id % (uint32_t)n_templates) * 64 : NULL;
        gco_env_init(&p->envs[i], board, agent_black, opponent, seed, id);
        p->envs[i].moves_max = moves_max; /* (only steps read it: the reset inside gco_env_init does not) */
    }
    return p;
}

gco_pool *gco_pool_new(uint64_t seed, uint32_t env_lo, uint32_t env_hi) {
    return gco_pool_new_cfg(seed, env_lo, env_hi, GCO_OPP_NONE, 0, 149, 0, NULL);
}

/* ChessEnvV2.reset of the envs with mask[i] != 0, as the CUDA env's masked reset does it: a new episode (so a BLACK
 * agent's opening ply is drawn with the new episode counter), the other envs keep their games */
void gco_pool_reset(gco_pool *p, const uint8_t *mask) {
    for (uint32_t i = 0; i < p->n; i++)
        if (mask[i]) {
            p->envs[i].episode++;
            gco_env_reset(&p->envs[i]);
        }
}

/* gco_env_view of every env: boards int8[n][64], info int32[n][16], legal uint16[n][stride] (the first min(n_legal,
 * stride) entries of a row are written) */
void gco_env_view(const gco_env *e, int8_t *board, int32_t *info, uint16_t *legal, int legal_cap);
void gco_pool_export(const gco_pool *p, int8_t *boards, int32_t *info, uint16_t *legal, int stride) {
    for (uint32_t i = 0; i < p->n; i++)
        gco_env_view(&p->envs[i], boards + (size_t)i * 64, info + (size_t)i * 16, legal + (size_t)i * (size_t)stride, stride);
}

static void pool_run(gco_pool *p, uint64_t nsteps_per_env, uint32_t stagger, int threads, gco_stats *st);
void gco_pool_run(gco_pool *p, uint64_t nsteps_per_env, int threads, gco_stats *st) {
    pool_run(p, nsteps_per_env, 0, threads, st);
}
/* env i runs nsteps_per_env + (i % stagger) steps: 3 random self-play episodes in 4 end at the 150-move cap after exactly 301
 * steps, so a pool started together stays in lockstep unless its phases are spread once */
void gco_pool_run_staggered(gco_pool *p, uint64_t nsteps_per_env, uint32_t stagger, int threads, gco_stats *st) {
    pool_run(p, nsteps_per_env, stagger, threads, st);
}
static void pool_run(gco_pool *p, uint64_t nsteps_per_env, uint32_t stagger, int threads, gco_stats *st) {
    if (threads < 1) threads = 1;
    if ((uint32_t)threads > p->n) threads = (int)(p->n ? p->n : 1);
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
    pool_arg *args = (pool_arg *)malloc(sizeof(pool_arg) * (size_t)threads);
    for (int t = 0; t < threads; t++) {
        args[t].pool = p, args[t].nsteps = nsteps_per_env, args[t].stagger = stagger;
        args[t].lo = (uint32_t)((uint64_t)p->n * (uint64_t)t / (uint64_t)threads);
        args[t].hi = (uint32_t)((uint64_t)p->n * (uint64_t)(t + 1) / (uint64_t)threads);
        pthread_create(&th[t], NULL, pool_worker, &args[t]);
    }
    memset(st, 0, sizeof(*st));
    for (int t = 0; t < threads; t++) {
        pthread_join(th[t], NULL);
        stats_add(st, &args[t].st);
    }
    free(th);
    free(args);
}

void gco_pool_free(gco_pool *p) {
    if (!p) return;
    for (uint32_t i = 0; i < p->n; i++) gco_env_free(&p->envs[i]);
    free(p->envs);
    free(p);
}

/* ------------------------------------------------------------------ batch wrappers (array in / array out) */

/* n positions in the reference wire format: boards int8[n][64], players int8[n] (+1/-1),
 * rights uint8[n][4] = (wk,wq,bk,bq).  out uint16[n][stride], counts int32[n] (true count, may exceed stride). */
void gco_movegen_batch(int n, const int8_t *boards, const int8_t *players, const uint8_t *rights, int attack,
                       uint16_t *out, int stride, int32_t *counts) {
    uint16_t tmp[GCO_MAX_MOVES];
    for (int i = 0; i < n; i++) {
        gco_state s;
        const uint8_t *r = rights + (size_t)i * 4;
        gco_state_new(&s, boards + (size_t)i * 64, players[i], r[0], r[1], r[2], r[3]);
        int c = gco_get_possible_moves(&s, players[i], attack, tmp, GCO_MAX_MOVES);
        counts[i] = c;
        for (int k = 0; k < c && k < stride; k++) out[(size_t)i * stride + k] = tmp[k];
    }
}

/* batched ChessEngine.next_state: out_boards int8[n][64], out_rights uint8[n][4], out_checks uint8[n][2]=(wchk,bchk),
 * out_reward int32[n], out_status int8[n] (0 ok, -1 empty from-square, -2 bad action) */
void gco_next_state_batch(int n, const int8_t *boards, const int8_t *players, const uint8_t *rights,
                          const int32_t *actions, int8_t *out_boards, uint8_t *out_rights, uint8_t *out_checks,
                          int32_t *out_reward, int8_t *out_status) {
    for (int i = 0; i < n; i++) {
        gco_state s, o;
        const uint8_t *r = rights + (size_t)i * 4;
        int rew = 0, both = 0;
        gco_state_new(&s, boards + (size_t)i * 64, players[i], r[0], r[1], r[2], r[3]);
        int rc = gco_next_state(&s, players[i], actions[i], &o, &rew, &both);
        out_status[i] = (int8_t)(rc ? rc : (both ? 1 : 0)); /* 1: both kings in check afterwards (lib.rs:1442-1446) */
        if (rc) { o = s; gco_update_state(&o); rew = 0; } /* reference panics; defined here as: position unchanged */
        memcpy(out_boards + (size_t)i * 64, o.board, 64);
        out_rights[(size_t)i * 4 + 0] = o.wk, out_rights[(size_t)i * 4 + 1] = o.wq;
        out_rights[(size_t)i * 4 + 2] = o.bk, out_rights[(size_t)i * 4 + 3] = o.bq;
        out_checks[(size_t)i * 2 + 0] = o.wchk, out_checks[(size_t)i * 2 + 1] = o.bchk;
        out_reward[i] = rew;
    }
}

/* batched ChessEngine.update_state */
void gco_update_state_batch(int n, const int8_t *boards, const uint8_t *rights, uint8_t *out_rights,
                            uint8_t *out_checks) {
    for (int i = 0; i < n; i++) {
        gco_state s;
        const uint8_t *r = rights + (size_t)i * 4;
        gco_state_new(&s, boards + (size_t)i * 64, GCO_WHITE, r[0], r[1], r[2], r[3]);
        gco_update_state(&s);
        out_rights[(size_t)i * 4 + 0] = s.wk, out_rights[(size_t)i * 4 + 1] = s.wq;
        out_rights[(size_t)i * 4 + 2] = s.bk, out_rights[(size_t)i * 4 + 3] = s.bq;
        out_checks[(size_t)i * 2 + 0] = s.wchk, out_checks[(size_t)i * 2 + 1] = s.bchk;
    }
}

typedef struct {
    int lo, hi, attack, stride;
    const int8_t *boards, *players;
    const uint8_t *rights;
    uint16_t *out;
    int32_t *counts;
} mg_arg;

static void *mg_worker(void *p) {
    mg_arg *a = (mg_arg *)p;
    gco_movegen_batch(a->hi - a->lo, a->boards + (size_t)a->lo * 64, a->players + a->lo, a->rights + (size_t)a->lo * 4,
                      a->attack, a->out + (size_t)a->lo * a->stride, a->stride, a->counts + a->lo);
    return NULL;
}

/* pthread version of gco_movegen_batch (CPU baseline for the movegen metric) */
void gco_movegen_batch_mt(int n, const int8_t *boards, const int8_t *players, const uint8_t *rights, int attack,
                          uint16_t *out, int stride, int32_t *counts, int threads) {
    if (threads < 1) threads = 1;
    if (threads > n) threads = n > 0 ? n : 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
    mg_arg *args = (mg_arg *)malloc(sizeof(mg_arg) * (size_t)threads);
    for (int t = 0; t < threads; t++) {
        mg_arg a = {(int)((int64_t)n * t / threads), (int)((int64_t)n * (t + 1) / threads), attack, stride, boards,
                    players, rights, out, counts};
        args[t] = a;
        pthread_create(&th[t], NULL, mg_worker, &args[t]);
    }
    for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
    free(th);
    free(args);
}

/* heap helpers so Python never needs to know sizeof(gco_env) */
gco_env *gco_env_new(const int8_t *initial_board, int agent_black, int opponent, uint64_t seed, uint32_t env_id) {
    gco_env *e = (gco_env *)malloc(sizeof(gco_env));
    gco_env_init(e, initial_board, agent_black, opponent, seed, env_id);
    return e;
}
void gco_env_delete(gco_env *e) {
    if (e) {
        gco_env_free(e);
        free(e);
    }
}
/* flat view of an env for comparisons: board[64], then
 * info[16] = {current_player, wk, wq, bk, bq, wchk, bchk, done, move_count, n_legal, episode, step_in_episode,
 *             last_bot_action, wedged_bot, hist_n, 0} */
void gco_env_view(const gco_env *e, int8_t *board, int32_t *info, uint16_t *legal, int legal_cap) {
    memcpy(board, e->st.board, 64);
    info[0] = e->st.current_player, info[1] = e->st.wk, info[2] = e->st.wq, info[3] = e->st.bk, info[4] = e->st.bq;
    info[5] = e->st.wchk, info[6] = e->st.bchk, info[7] = e->done, info[8] = e->move_count, info[9] = e->n_legal;
    info[10] = (int32_t)e->episode, info[11] = (int32_t)e->step_in_episode, info[12] = e->last_bot_action;
    info[13] = e->wedged_bot, info[14] = e->hist_n, info[15] = 0;
    for (int k = 0; k < e->n_legal && k < legal_cap; k++) legal[k] = e->legal[k];
}
void gco_env_set_episode(gco_env *e, uint32_t episode) { e->episode = episode; }
/* ChessEnvV2.moves_max (chess_v2.py:141) is a plain attribute: 149 unless the user changes it */
void gco_env_set_moves_max(gco_env *e, int moves_max) { e->moves_max = moves_max; }
void gco_env_force_bot(gco_env *e, int action) { e->forced_bot_action = action; }
/* A new episode from an arbitrary state (what assigning `env.state = s` -- the setter of chess_v2.py:315-323 -- plus the
 * bookkeeping of reset() amounts to): engine.update_state masks the flags and computes the check flags, then
 * get_possible_moves for the side to move.  The episode counter is set by the caller (gco_env_set_episode). */
void gco_env_import(gco_env *e, const int8_t *board, int player, int wk, int wq, int bk, int bq, int move_count) {
    e->done = 0;
    e->hist_n = 0;
    e->move_count = move_count;
    e->wedged_bot = 0;
    e->step_in_episode = 0;
    e->last_bot_action = -1;
    gco_state_new(&e->st, board, player, wk, wq, bk, bq);
    gco_update_state(&e->st);
    env_movegen(e, player);
}
