/* TEST INFRASTRUCTURE ONLY (tests/test_edit_records.py compiles it into a temporary directory).
 *
 * gpo_ntedit_contig of the C restatement (oracle/gp_oracle.c, included unchanged below) that also writes where every
 * output byte came from, for the edit records of gp_polish_fetch_edits: origin[o] = the position in seq_in of the input
 * byte that output byte o copies, or NTEDIT_INSERTED for a byte the rope inserted -- the rule of the edit kernel's
 * emit_rope.  The edit loop is a copy of gpo_ntedit_contig's; only the FASTA-body loop at the end adds the origins.
 */
#include "../oracle/gp_oracle.c"

#define NTEDIT_INSERTED 0xFFFFFFFFu

long ntedit_contig_origins(const char* seq_in, size_t len, const uint8_t* bf, size_t bf_bytes,
                           const gpo_ntedit_opts* opts, char* outbuf, size_t cap, gpo_ntedit_stats* stats,
                           uint32_t* origin)
{
  if (len < opts->min_contig_len) return -1; /* readAndCorrect, :1850 */
  ed_t E;
  memset(&E, 0, sizeof E);
  ed_t* e = &E;
  e->o = *opts;
  e->seq = (char*)malloc(len + 1);
  memcpy(e->seq, seq_in, len);
  e->seq[len] = 0;
  e->len = (uint32_t)len;
  e->bf = bf;
  e->bf_bits = (uint64_t)bf_bytes * 8ULL;
  e->insertion_cap = (unsigned)((float)opts->k * 1.5f); /* :2024-2025 */
  /* float thresholds exactly as written at :1521-1523, :1624-1626 / :1335-1337, :1228-1230 */
  e->thr_missing = ((float)opts->k / (float)opts->jump) * opts->missing_ratio;
  e->thr_edit = ((float)opts->k / (float)opts->jump) * opts->edit_ratio;
  e->thr_del = (1 + ((float)opts->k / (float)opts->jump)) * opts->edit_ratio;
  const uint32_t k = opts->k;

  hstate_t hs = { 0, 0 };
  unsigned char char_in = 0, char_out = 0;
  cursor_t c;
  c.h_seq = find_first_accepted_kmer(e, 0);
  c.t_seq = c.h_seq + k - 1;
  if ((uint64_t)c.h_seq + k - 1 < len) { /* :1441-1444 */
    hs.fh = gpo_ntf64(e->seq + c.h_seq, k);
    hs.rh = gpo_ntr64(e->seq + c.h_seq, k);
    char_in = (unsigned char)e->seq[c.t_seq];
  }
  node_t root = { 0, 0, (uint32_t)len - 1, 0 };
  nodes_set(e, 0, root);
  c.h_node = c.t_node = 0;

  int continue_edit = 1;
  do {
    if ((uint64_t)c.h_seq + k - 1 >= len) break; /* :1463 */
    if (!bf_contains(e, &hs)) {                /* :1470 */
      e->st.triggers++;
      cursor_t tc = c;
      hstate_t th = hs;
      const unsigned char draft_char = (unsigned char)toupper(char_in); /* :1480 */
      unsigned check_missing = 0;
      int do_not_fix = 0;
      for (unsigned kk = 0; kk < k && tc.h_seq < len; kk++) { /* :1487-1512 */
        if (roll(e, &tc, &char_out, &char_in)) {
          hs_roll(e, &th, char_out, char_in);
          if (!is_accepted(char_in)) { do_not_fix = 1; break; }
          if (kk % opts->jump == 0 && !bf_contains(e, &th)) check_missing++;
        } else { do_not_fix = 1; break; }
      }
      if (!do_not_fix && (float)check_missing >= e->thr_missing) { /* :1517-1523 */
        e->st.attempts++;
        unsigned num_deletions = 1; /* :1526 */
        best_t best;
        memset(&best, 0, sizeof best);
        unsigned char bases[4];
        const int nb = polish_bases(draft_char, bases);
        for (int b = 0; b < nb; b++) { /* :1559-1713 */
          const unsigned char sub_base = bases[b];
          th = hs;
          hs_changelast(e, &th, draft_char, sub_base);
          if (!bf_contains(e, &th) && opts->mode != 2) continue; /* :1569-1570 */
          tc = c;
          const node_t tn = e->nodes[c.t_node];
          if (tn.type == 0) e->seq[tc.t_seq] = (char)sub_base; /* :1578-1582 */
          else if (tn.type == 1) e->nodes[c.t_node].c = sub_base;
          unsigned present = 0;
          for (unsigned kk = 0; kk < k && tc.h_seq < len && tc.t_seq < len; kk++) { /* :1585-1606 */
            if (roll(e, &tc, &char_out, &char_in)) {
              hs_roll(e, &th, char_out, char_in);
              if (kk % opts->jump == 0 && bf_contains(e, &th)) present++;
            } else break;
          }
          if (tn.type == 0) e->seq[c.t_seq] = (char)draft_char; /* revert with the UPPER-cased char, :1609-1615 */
          else if (tn.type == 1) e->nodes[c.t_node].c = draft_char;
          if ((float)present >= e->thr_edit) { /* :1621-1626 */
            if (present >= best.support) {   /* :1629 (>= : later base wins ties) */
              best.type = 1; best.sub_base = sub_base; best.support = present;
            }
            if (opts->mode == 0 || opts->mode == 1) continue; /* :1680-1682 */
          }
          if (opts->mode == 2 || best.type != 1) { /* :1686 */
            if (try_indels(e, draft_char, sub_base, &num_deletions, &c, &hs, &best)) {
              if (opts->mode == 0 || opts->mode == 1) break; /* :1707-1709 */
            }
          }
        }
        make_edit(e, draft_char, &best, &c, &hs); /* :1715-1736 */
      }
    }
    /* roll forward, skipping k past any non-accepted incoming char, :1740-1759 */
    long target = -1;
    do {
      if (roll(e, &c, &char_out, &char_in)) {
        if (!is_accepted(char_in)) target = (long)c.t_seq + (long)k;
        hs_roll(e, &hs, char_out, char_in);
      } else { continue_edit = 0; break; }
    } while (target >= 0 && (long)c.t_seq != target);
  } while (continue_edit);

  /* writeEditsToFile body, :797-935 */
  size_t o = 0;
  long rc = 0;
  for (size_t i = 0; i < e->n && e->nodes[i].type != -1; i++) {
    const node_t* nd = &e->nodes[i];
    if (nd->type == 0) {
      /* substr(s_pos, e_pos - s_pos + 1) with size_t arithmetic: e_pos < s_pos wraps to a
         huge count == "to the end of the string"; s_pos > size throws */
      size_t s = nd->s, cnt;
      if (s > len) { e->st.ref_ub++; continue; }
      if (nd->e + 1u >= nd->s) cnt = (size_t)nd->e + 1 - s; else cnt = len - s;
      if (s + cnt > len) cnt = len - s;
      if (o + cnt > cap) { rc = -2; break; }
      memcpy(outbuf + o, e->seq + s, cnt);
      for (size_t q = 0; q < cnt; q++) origin[o + q] = (uint32_t)(s + q);
      o += cnt;
    } else {
      if (o + 1 > cap) { rc = -2; break; }
      origin[o] = NTEDIT_INSERTED;
      outbuf[o++] = (char)nd->c;
    }
  }
  if (stats) *stats = e->st;
  free(e->seq);
  free(e->nodes);
  return rc < 0 ? rc : (long)o;
}
