/* The reference PipLib's example program (example/example.c: the only caller of the library inside the
 * reference tree, driven by its `make check` over the example .pip files), restated for the tests with the
 * same calls in the same order and the same output.  It reads, from stdin, the context matrix, the bignum
 * column, the constraint matrix and option keywords, echoes the input with prompts, solves with pip_solve
 * and prints the quast with pip_quast_print.  It uses only the public API, so it builds unchanged against
 * include/ and links with -lpiplib_dp: the drop-in claim checked as a C program (tests/test_cabi.py compiles
 * it, tests/test_gpu_parity.py runs it against the reference's golden .ll transcripts). */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <strings.h>
#include <unistd.h>

#include <piplib/piplib64.h>

int main(int argc, const char **argv)
{
  int bignum, verbose = 0;
  char line[1024];
  PipMatrix *domain, *context;
  PipQuast *solution;
  PipOptions *options;

  for (int i = 1; i < argc; i++)
    if (strcmp(argv[i], "-v") == 0)
      verbose++;

  printf("[PIP2-like future input] Please enter:\n- the context matrix,\n");
  context = pip_matrix_read(stdin);
  pip_matrix_print(stdout, context);

  printf("- the bignum column (start at 0, -1 if no bignum),\n");
  if (fscanf(stdin, " %d", &bignum) != 1)
    return 1;
  printf("%d\n", bignum);

  printf("- the constraint matrix.\n");
  domain = pip_matrix_read(stdin);
  pip_matrix_print(stdout, domain);
  printf("\n");

  if (isatty(0))
    printf("- options (EOF to stop).\n");
  options = pip_options_init();
  options->Verbose = verbose;
  while (fgets(line, sizeof line, stdin)) {
    if (strncasecmp(line, "Maximize", 8) == 0)
      options->Maximize = 1;
    if (strncasecmp(line, "Urs_parms", 9) == 0)
      options->Urs_parms = 1;
    if (strncasecmp(line, "Urs_unknowns", 12) == 0)
      options->Urs_unknowns = 1;
    if (strncasecmp(line, "Rational", 8) == 0)
      options->Nq = 0;
    if (strncasecmp(line, "Dual", 4) == 0)
      options->Compute_dual = 1;
  }

  /* the bignum column is counted in the context; the library wants it in the whole tableau */
  if (bignum > 0)
    bignum += domain->NbColumns - context->NbColumns;
  solution = pip_solve(domain, context, bignum, options);

  pip_options_free(options);
  pip_matrix_free(domain);
  pip_matrix_free(context);

  pip_quast_print(stdout, solution, 0);
  pip_quast_free(solution);
  return 0;
}
