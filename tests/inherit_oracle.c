/*
 * inherit_oracle.c — CPU restatement of the de novo rule with inheritance (DESIGN.md §2
 * "Inheritance"), test infrastructure only.  orc_calls_inherit is oracle/dnk_oracle.c's
 * orc_calls with only the clauses of the parents who can transmit the variant's locus to the
 * child: cls[v] 0 autosomal (PARs included), 1 X, 2 Y (both outside the PARs), 3 mitochondrial
 * (cls NULL: all autosomal); sex 0 unknown, 1 male, 2 female.  The table below is written out
 * as DESIGN.md prints it and shares nothing with the CUDA path; tests/inherit_oracle.py pins it
 * against a pure-Python reading of the same table.
 */
#include <stdint.h>
#include <stddef.h>
#include <string.h>

/* Row: locus class; column: the child's sex.  'M' = the mother's clauses apply, 'F' = the
 * father's; "-" = neither does and the child has no copy of the locus (bit 0x20). */
static const char *const PARENTS[4][3] = {
    /*              unknown  male  female */
    /* autosomal */ {"MF", "MF", "MF"},
    /* X         */ {"MF", "M", "MF"},
    /* Y         */ {"MF", "F", "-"},
    /* maternal  */ {"M", "M", "M"},
};

/* hits / distinct: [n_variants][2 alleles][3 samples: child, mother, father], as orc_calls. */
void orc_calls_inherit(const uint64_t *hits, const uint64_t *distinct, size_t n_variants,
                       uint32_t min_child_alt_hits, uint32_t min_child_alt_distinct,
                       uint32_t max_parent_alt_hits, uint32_t min_parent_ref_hits, const uint8_t *cls,
                       uint8_t sex, uint8_t *calls) {
  for (size_t v = 0; v < n_variants; v++) {
    const char *who = PARENTS[cls ? cls[v] : 0][sex];
    const int mother = strchr(who, 'M') != NULL, father = strchr(who, 'F') != NULL;
    const uint64_t *ref = hits + v * 6, *alt = hits + v * 6 + 3, *alt_d = distinct + v * 6 + 3;
    uint8_t c = 0;
    if (alt[0] < min_child_alt_hits || alt_d[0] < min_child_alt_distinct) c |= 0x02;
    if (mother && alt[1] > max_parent_alt_hits) c |= 0x04;
    if (father && alt[2] > max_parent_alt_hits) c |= 0x08;
    if ((mother && ref[1] < min_parent_ref_hits) || (father && ref[2] < min_parent_ref_hits)) c |= 0x10;
    if (who[0] == '-') c |= 0x20;
    calls[v] = c ? c : 0x01;
  }
}
