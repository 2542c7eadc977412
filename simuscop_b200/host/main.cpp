// main.cpp -- drop-in `simuReads <configuration file>` (reference src/simuReads.cpp:24-97).
// New knobs come from the environment only, so existing configuration files stay valid:
//   SIMUSCOP_SEED (default: wall clock, like the reference), SIMUSCOP_DEVICE (default 0),
//   SIMUSCOP_DUMP_PLAN=<prefix>, SIMUSCOP_BATCH_PAIRS, SIMUSCOP_GZIP=1 (<name>.fq.gz, compressed on the GPU),
//   SIMUSCOP_BGZF=1 (<name>.fq.gz as BGZF blocks + its <name>.fq.gz.gzi index: parallel decompression, random access),
//   SIMUSCOP_INTERLEAVE=1 (PE: one <name>.fq, mates in turn), SIMUSCOP_BAM=1 (<name>.bam: unaligned BAM, read group
//   <name>, PE and SE; before SIMUSCOP_GZIP / BGZF / INTERLEAVE), SIMUSCOP_STDOUT=1 (the reads to standard output, e.g.
//   `simuReads config | bwa mem -p ref.fa -`).  Every message goes to stderr, so stdout carries FASTQ or BAM bytes only.
#include <signal.h>

#include <chrono>
#include <cstdlib>
#include <ctime>
#include <iostream>

#include "../../include/simuscop_host.h"

static void usage(const char* app) {
	std::cerr << "\nVersion: simuscop-b200 1.0 (B200-native simuReads)\n\n"
	          << "Usage: " << app << " <configuration file>\n\n"
	          << "Example:\n    " << app << " /path/to/config.txt\n" << std::endl;
}

int main(int argc, char* argv[]) {
	if (argc == 1) { std::cerr << "Error: configuration file is required!" << std::endl; usage(argv[0]); return 1; }
	if (argc > 2) { std::cerr << "Error: too many input arguments!" << std::endl; usage(argv[0]); return 1; }
	time_t start_t = time(NULL);
	const char* s = getenv("SIMUSCOP_SEED");
	uint64_t seed = s ? strtoull(s, NULL, 10) : (uint64_t)std::chrono::system_clock::now().time_since_epoch().count();
	const char* d = getenv("SIMUSCOP_DEVICE");
	// a reader that closes the pipe early makes the next write fail with EPIPE instead of killing the process: the run ends
	// with an error message and exit code 1
	const char* so = getenv("SIMUSCOP_STDOUT");
	if (so && atoi(so) != 0) signal(SIGPIPE, SIG_IGN);
	ssh_job* job = nullptr;
	if (ssh_open(argv[1], seed, &job)) return 1;
	int rc = ssh_run(job, d ? atoi(d) : 0);
	ssh_close(job);
	if (rc) return 1;
	std::cerr << "\nReads generation done!" << std::endl;
	long used = (long)(time(NULL) - start_t);
	std::cerr << "\nElapsed time: " << used / 60 << " minutes and " << used % 60 << " seconds!\n" << std::endl;
	return 0;
}
