/* TEST INFRASTRUCTURE -- not product code.
 *
 * ref_dump.c (the recording driver around the unmodified reference producer) with one more switch:
 *   --almanac    sim.almanac_enable = true, as the reference program has it by default (gps-sim.c:189).
 *                The producer then reads almanac.sem from the WORKING DIRECTORY (almanac.c:87) and fills the
 *                almanac pages of subframes 4 and 5 (gps.c:772-884).
 * Every other switch is ref_dump.c's; without --almanac the binary behaves exactly like ref_dump.
 *
 * ref_dump.c is compiled as is: its main() becomes ref_dump_main(), and its one pthread_create() call -- the start
 * of gps_thread_ep on its simulator_t -- goes through oracle_start_producer(), which sets the flag first. The
 * reference sources do not call pthread_create themselves.
 */
#include <pthread.h>
#include <stdbool.h>
#include <string.h>

static bool g_almanac;

static int oracle_start_producer(pthread_t *th, const pthread_attr_t *attr, void *(*fn)(void *), void *arg);

#define main ref_dump_main
#define pthread_create oracle_start_producer
#include "ref_dump.c"
#undef pthread_create
#undef main

static int oracle_start_producer(pthread_t *th, const pthread_attr_t *attr, void *(*fn)(void *), void *arg) {
    if (fn == gps_thread_ep) ((simulator_t *) arg)->almanac_enable = g_almanac;
    return pthread_create(th, attr, fn, arg);
}

int main(int argc, char **argv) {
    int n = 0;
    for (int i = 0; i < argc; i++) {
        if (i > 0 && !strcmp(argv[i], "--almanac")) g_almanac = true;
        else argv[n++] = argv[i];
    }
    argv[n] = NULL;
    return ref_dump_main(n, argv);
}
