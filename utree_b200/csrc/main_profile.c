/* main_profile.c -- `utree-profile`: reads per taxonomy string for one or more samples, as one TSV table
 * (utb_profile_main, include/utree_b200.h). */
#include "../../include/utree_b200.h"
int main(int argc, char **argv) { return utb_profile_main(argc, argv); }
