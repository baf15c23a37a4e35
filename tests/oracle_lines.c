/*
 * tests/oracle_lines.c — TEST INFRASTRUCTURE ONLY.
 *
 * The line records of ugx_find_lines restated on top of the oracle (oracle/oracle.c, included whole so that its
 * find loop is reused as it stands): tests/lines_oracle.py compiles this file into a shared library of its own.
 */
#include "../oracle/oracle.c"

int ora_find_lines(const ora_pattern *p, const uint8_t *buf, uint64_t n, uint64_t base_offset, uint64_t base_line,
                   int invert, ugx_line *out, uint64_t cap, uint64_t *n_out);

/*
 * Line records: the `ugrep -c` loop (ora_count_lines) recording the match each find() returns, with the line it lies on
 * (lineno(), and bol() / eol() of that line: the '\n' after it, or the buffer end); with `invert` the other lines, in
 * order, offset = bol, len = cap = 0.  The lines of a buffer are its newlines, plus one when it does not end in '\n'.
 */
int ora_find_lines(const ora_pattern *p, const uint8_t *buf, uint64_t n, uint64_t base_offset, uint64_t base_line,
                   int invert, ugx_line *out, uint64_t cap, uint64_t *n_out)
{
  scan_t m;
  scan_init(&m, p, buf, n);
  uint64_t c = 0;
  uint64_t lno = 1;  /* lineno() of position `at` */
  size_t bol = 0;    /* start of that line */
  size_t at = 0;
  int hit_line = 0;  /* the line at `at` has a match */
  uint32_t acc;
  for (;;)
  {
    acc = match_find(&m);
    const size_t to = acc != 0 ? m.txt : (size_t)n;
    for (; at < to; ++at)
      if (buf[at] == '\n')
      {
        if (invert && !hit_line)
        {
          if (c < cap)
          {
            out[c].line = lno + base_line;
            out[c].bol = bol + base_offset;
            out[c].eol = at + base_offset;
            out[c].offset = bol + base_offset;
            out[c].len = 0;
            out[c].cap = 0;
          }
          ++c;
        }
        ++lno;
        bol = at + 1;
        hit_line = 0;
      }
    if (acc == 0)
      break;
    if (!invert)
    {
      size_t eol = m.txt;
      while (eol < n && buf[eol] != '\n')
        ++eol;
      if (c < cap)
      {
        out[c].line = lno + base_line;
        out[c].bol = bol + base_offset;
        out[c].eol = eol + base_offset;
        out[c].offset = m.txt + base_offset;
        out[c].len = (uint32_t)m.len;
        out[c].cap = acc;
      }
      ++c;
    }
    hit_line = 1;
    if (m.got != '\n') /* !at_bol(): src/ugrep.cpp:10583-10584 */
      skip_newline(&m);
  }
  /* an unterminated last line */
  if (invert && !hit_line && bol < n)
  {
    if (c < cap)
    {
      out[c].line = lno + base_line;
      out[c].bol = bol + base_offset;
      out[c].eol = n + base_offset;
      out[c].offset = bol + base_offset;
      out[c].len = 0;
      out[c].cap = 0;
    }
    ++c;
  }
  *n_out = c;
  return c > cap ? UGX_E_OVERFLOW : UGX_OK;
}

