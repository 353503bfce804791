/* main.c -- minimap2-compatible command line for the B200 build.
 * Same option letters, long options, two-pass preset handling and defaults as the reference CLI
 * (main.c:32-85,111-286; mapping flow :346-399 in its de-instrumented form), parsed with getopt_long.
 * Extra: --gpus INT (GPUs of this node to use; the index is replicated to each). */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <errno.h>
#include <getopt.h>
#include <sys/resource.h>
#include "minimap_b200.h"

#define MM_VERSION "2.17-r954-b200"
#define MM_DBG_NO_KALLOC 0x1
#define MM_DBG_PRINT_QNAME 0x2
#define MM_DBG_PRINT_SEED 0x4
#define MM_DBG_PRINT_ALN_SEQ 0x8

extern double realtime(void), cputime(void);
extern long peakrss(void);

static struct option long_options[] = {
	{ "bucket-bits",    required_argument, 0, 300 }, { "mb-size",        required_argument, 0, 'K' },
	{ "seed",           required_argument, 0, 302 }, { "no-kalloc",      no_argument,       0, 303 },
	{ "print-qname",    no_argument,       0, 304 }, { "no-self",        no_argument,       0, 'D' },
	{ "print-seeds",    no_argument,       0, 306 }, { "max-chain-skip", required_argument, 0, 307 },
	{ "min-dp-len",     required_argument, 0, 308 }, { "print-aln-seq",  no_argument,       0, 309 },
	{ "splice",         no_argument,       0, 310 }, { "cost-non-gt-ag", required_argument, 0, 'C' },
	{ "no-long-join",   no_argument,       0, 312 }, { "sr",             no_argument,       0, 313 },
	{ "frag",           required_argument, 0, 314 }, { "secondary",      required_argument, 0, 315 },
	{ "cs",             optional_argument, 0, 316 }, { "end-bonus",      required_argument, 0, 317 },
	{ "no-pairing",     no_argument,       0, 318 }, { "splice-flank",   required_argument, 0, 319 },
	{ "idx-no-seq",     no_argument,       0, 320 }, { "end-seed-pen",   required_argument, 0, 321 },
	{ "for-only",       no_argument,       0, 322 }, { "rev-only",       no_argument,       0, 323 },
	{ "heap-sort",      required_argument, 0, 324 }, { "all-chain",      no_argument,       0, 'P' },
	{ "dual",           required_argument, 0, 326 }, { "max-clip-ratio", required_argument, 0, 327 },
	{ "min-occ-floor",  required_argument, 0, 328 }, { "MD",             no_argument,       0, 329 },
	{ "lj-min-ratio",   required_argument, 0, 330 }, { "score-N",        required_argument, 0, 331 },
	{ "eqx",            no_argument,       0, 332 }, { "paf-no-hit",     no_argument,       0, 333 },
	{ "split-prefix",   required_argument, 0, 334 }, { "no-end-flt",     no_argument,       0, 335 },
	{ "hard-mask-level",no_argument,       0, 336 }, { "cap-sw-mem",     required_argument, 0, 337 },
	{ "max-qlen",       required_argument, 0, 338 }, { "max-chain-iter", required_argument, 0, 339 },
	{ "junc-bed",       required_argument, 0, 340 }, { "junc-bonus",     required_argument, 0, 341 },
	{ "sam-hit-only",   no_argument,       0, 342 }, { "gpus",           required_argument, 0, 400 },
	{ "help",           no_argument,       0, 'h' }, { "max-intron-len", required_argument, 0, 'G' },
	{ "version",        no_argument,       0, 'V' }, { "min-count",      required_argument, 0, 'n' },
	{ "min-chain-score",required_argument, 0, 'm' }, { "mask-level",     required_argument, 0, 'M' },
	{ "min-dp-score",   required_argument, 0, 's' }, { "sam",            no_argument,       0, 'a' },
	{ 0, 0, 0, 0 }
};

static int64_t parse_num(const char *str)
{ /* 4G / 500M / 10k suffixes (main.c:87-97) */
	char *p;
	double x = strtod(str, &p);
	if (*p == 'G' || *p == 'g') x *= 1e9;
	else if (*p == 'M' || *p == 'm') x *= 1e6;
	else if (*p == 'K' || *p == 'k') x *= 1e3;
	return (int64_t)(x + .499);
}

static void yes_or_no(mm_mapopt_t *opt, int64_t flag, const char *name, const char *arg, int yes_to_set)
{
	const int yes = !strcmp(arg, "yes") || !strcmp(arg, "y"), no = !strcmp(arg, "no") || !strcmp(arg, "n");
	if (!yes && !no) { fprintf(stderr, "[WARNING]\033[1;31m option '--%s' only accepts 'yes' or 'no'.\033[0m\n", name); return; }
	if (yes == !!yes_to_set) opt->flag |= flag;
	else opt->flag &= ~flag;
}

static void usage(FILE *fp, const mm_idxopt_t *ipt, const mm_mapopt_t *opt, int n_threads)
{
	fprintf(fp, "Usage: minimap2 [options] <target.fa> [query.fa] [...]\n");
	fprintf(fp, "Options:\n  Indexing:\n");
	fprintf(fp, "    -H           use homopolymer-compressed k-mer (preferrable for PacBio)\n");
	fprintf(fp, "    -k INT       k-mer size (no larger than 28) [%d]\n", ipt->k);
	fprintf(fp, "    -w INT       minimizer window size [%d]\n", ipt->w);
	fprintf(fp, "    -I NUM       split index for every ~NUM input bases [4G]\n");
	fprintf(fp, "  Mapping:\n");
	fprintf(fp, "    -f FLOAT     filter out top FLOAT fraction of repetitive minimizers [%g]\n", opt->mid_occ_frac);
	fprintf(fp, "    -g NUM       stop chain enlongation if there are no minimizers in INT-bp [%d]\n", opt->max_gap);
	fprintf(fp, "    -G NUM       max intron length (effective with -xsplice; changing -r) [200k]\n");
	fprintf(fp, "    -F NUM       max fragment length (effective with -xsr or in the fragment mode) [800]\n");
	fprintf(fp, "    -r NUM       bandwidth used in chaining and DP-based alignment [%d]\n", opt->bw);
	fprintf(fp, "    -n INT       minimal number of minimizers on a chain [%d]\n", opt->min_cnt);
	fprintf(fp, "    -m INT       minimal chaining score (matching bases minus log gap penalty) [%d]\n", opt->min_chain_score);
	fprintf(fp, "    -X           skip self and dual mappings (for the all-vs-all mode)\n");
	fprintf(fp, "    -p FLOAT     min secondary-to-primary score ratio [%g]\n", opt->pri_ratio);
	fprintf(fp, "    -N INT       retain at most INT secondary alignments [%d]\n", opt->best_n);
	fprintf(fp, "  Alignment:\n");
	fprintf(fp, "    -A INT       matching score [%d]\n", opt->a);
	fprintf(fp, "    -B INT       mismatch penalty [%d]\n", opt->b);
	fprintf(fp, "    -O INT[,INT] gap open penalty [%d,%d]\n", opt->q, opt->q2);
	fprintf(fp, "    -E INT[,INT] gap extension penalty; a k-long gap costs min{O1+k*E1,O2+k*E2} [%d,%d]\n", opt->e, opt->e2);
	fprintf(fp, "    -z INT[,INT] Z-drop score and inversion Z-drop score [%d,%d]\n", opt->zdrop, opt->zdrop_inv);
	fprintf(fp, "    -s INT       minimal peak DP alignment score [%d]\n", opt->min_dp_max);
	fprintf(fp, "  Input/Output:\n");
	fprintf(fp, "    -a           output in the SAM format (PAF by default)\n");
	fprintf(fp, "    -o FILE      output alignments to FILE [stdout]\n");
	fprintf(fp, "    -L           write CIGAR with >65535 ops at the CG tag\n");
	fprintf(fp, "    -R STR       SAM read group line in a format like '@RG\\tID:foo\\tSM:bar' []\n");
	fprintf(fp, "    -c           output CIGAR in PAF\n");
	fprintf(fp, "    --cs[=STR]   output the cs tag; STR is 'short' (if absent) or 'long' [none]\n");
	fprintf(fp, "    --MD         output the MD tag\n");
	fprintf(fp, "    --eqx        write =/X CIGAR operators\n");
	fprintf(fp, "    -Y           use soft clipping for supplementary alignments\n");
	fprintf(fp, "    -t INT       number of host threads [%d]\n", n_threads);
	fprintf(fp, "    --gpus INT   number of GPUs to use [1]\n");
	fprintf(fp, "    -K NUM       minibatch size for mapping [500M]\n");
	fprintf(fp, "    --version    show version number\n");
	fprintf(fp, "  Preset:\n");
	fprintf(fp, "    -x STR       preset (always applied before other options) []\n");
	fprintf(fp, "                 - map-pb/map-ont: PacBio/Nanopore vs reference mapping\n");
	fprintf(fp, "                 - sr: genomic short-read mapping\n");
}

int main(int argc, char *argv[])
{
	const char *opt_str = "2aSDw:k:K:t:r:f:Vv:g:G:I:d:XT:s:x:Hcp:M:n:z:A:B:O:E:m:N:Qu:R:hF:LC:yYPo:";
	mm_mapopt_t opt;
	mm_idxopt_t ipt;
	int i, c, n_threads = 3, old_best_n = -1, n_gpus = 1, longidx = -1;
	char *fnw = 0, *rg = 0, *s;
	FILE *fp_help = stderr;
	mm_idx_reader_t *idx_rdr;
	mm_idx_t *mi;
	struct rlimit rl;
	char **argv0 = (char**)malloc((size_t)(argc + 1) * sizeof(char*)); /* getopt_long permutes argv; the @PG line shows the original */

	memcpy(argv0, argv, (size_t)(argc + 1) * sizeof(char*));
	mm_verbose = 3;
	getrlimit(RLIMIT_AS, &rl); rl.rlim_cur = rl.rlim_max; setrlimit(RLIMIT_AS, &rl);
	mm_realtime0 = realtime();
	mm_set_opt(0, &ipt, &opt);

	opterr = 0;
	while ((c = getopt_long(argc, argv, opt_str, long_options, 0)) >= 0) { /* presets first */
		if (c == 'x') {
			if (mm_set_opt(optarg, &ipt, &opt) < 0) { fprintf(stderr, "[ERROR] unknown preset '%s'\n", optarg); return 1; }
		} else if (c == ':') { fprintf(stderr, "[ERROR] missing option argument\n"); return 1; }
		else if (c == '?') { fprintf(stderr, "[ERROR] unknown option in \"%s\"\n", argv[optind - 1]); return 1; }
	}
	optind = 0;
	while ((c = getopt_long(argc, argv, opt_str, long_options, &longidx)) >= 0) {
		const char *lname = longidx >= 0 ? long_options[longidx].name : "";
		if (c == 'w') ipt.w = atoi(optarg);
		else if (c == 'k') ipt.k = atoi(optarg);
		else if (c == 'H') ipt.flag |= MM_I_HPC;
		else if (c == 'd') fnw = optarg;
		else if (c == 'r') opt.bw = (int)parse_num(optarg);
		else if (c == 't') n_threads = atoi(optarg);
		else if (c == 'v') mm_verbose = atoi(optarg);
		else if (c == 'g') opt.max_gap = (int)parse_num(optarg);
		else if (c == 'G') mm_mapopt_max_intron_len(&opt, (int)parse_num(optarg));
		else if (c == 'F') opt.max_frag_len = (int)parse_num(optarg);
		else if (c == 'N') old_best_n = opt.best_n, opt.best_n = atoi(optarg);
		else if (c == 'p') opt.pri_ratio = atof(optarg);
		else if (c == 'M') opt.mask_level = atof(optarg);
		else if (c == 'c') opt.flag |= MM_F_OUT_CG | MM_F_CIGAR;
		else if (c == 'D') opt.flag |= MM_F_NO_DIAG;
		else if (c == 'P') opt.flag |= MM_F_ALL_CHAINS;
		else if (c == 'X') opt.flag |= MM_F_ALL_CHAINS | MM_F_NO_DIAG | MM_F_NO_DUAL | MM_F_NO_LJOIN;
		else if (c == 'a') opt.flag |= MM_F_OUT_SAM | MM_F_CIGAR;
		else if (c == 'Q') opt.flag |= MM_F_NO_QUAL;
		else if (c == 'Y') opt.flag |= MM_F_SOFTCLIP;
		else if (c == 'L') opt.flag |= MM_F_LONG_CIGAR;
		else if (c == 'y') opt.flag |= MM_F_COPY_COMMENT;
		else if (c == 'T') opt.sdust_thres = atoi(optarg);
		else if (c == 'n') opt.min_cnt = atoi(optarg);
		else if (c == 'm') opt.min_chain_score = atoi(optarg);
		else if (c == 'A') opt.a = atoi(optarg);
		else if (c == 'B') opt.b = atoi(optarg);
		else if (c == 's') opt.min_dp_max = atoi(optarg);
		else if (c == 'C') opt.noncan = atoi(optarg);
		else if (c == 'I') ipt.batch_size = parse_num(optarg);
		else if (c == 'K') opt.mini_batch_size = (int)parse_num(optarg);
		else if (c == 'R') rg = optarg;
		else if (c == 'h') fp_help = stdout;
		else if (c == '2') opt.flag |= MM_F_2_IO_THREADS;
		else if (c == 'o') {
			if (strcmp(optarg, "-") != 0 && freopen(optarg, "wb", stdout) == NULL) {
				fprintf(stderr, "[ERROR]\033[1;31m failed to write the output to file '%s'\033[0m: %s\n", optarg, strerror(errno));
				exit(1);
			}
		}
		else if (c == 300) ipt.bucket_bits = atoi(optarg);
		else if (c == 302) opt.seed = atoi(optarg);
		else if (c == 303) mm_dbg_flag |= MM_DBG_NO_KALLOC;
		else if (c == 304) mm_dbg_flag |= MM_DBG_PRINT_QNAME;
		else if (c == 306) mm_dbg_flag |= MM_DBG_PRINT_QNAME | MM_DBG_PRINT_SEED, n_threads = 1;
		else if (c == 307) opt.max_chain_skip = atoi(optarg);
		else if (c == 339) opt.max_chain_iter = atoi(optarg);
		else if (c == 308) opt.min_ksw_len = atoi(optarg);
		else if (c == 309) mm_dbg_flag |= MM_DBG_PRINT_QNAME | MM_DBG_PRINT_ALN_SEQ, n_threads = 1;
		else if (c == 310) opt.flag |= MM_F_SPLICE;
		else if (c == 312) opt.flag |= MM_F_NO_LJOIN;
		else if (c == 313) opt.flag |= MM_F_SR;
		else if (c == 317) opt.end_bonus = atoi(optarg);
		else if (c == 318) opt.flag |= MM_F_INDEPEND_SEG;
		else if (c == 320) ipt.flag |= MM_I_NO_SEQ;
		else if (c == 321) opt.anchor_ext_shift = atoi(optarg);
		else if (c == 322) opt.flag |= MM_F_FOR_ONLY;
		else if (c == 323) opt.flag |= MM_F_REV_ONLY;
		else if (c == 327) opt.max_clip_ratio = atof(optarg);
		else if (c == 328) opt.min_mid_occ = atoi(optarg);
		else if (c == 329) opt.flag |= MM_F_OUT_MD;
		else if (c == 330) opt.min_join_flank_ratio = atof(optarg);
		else if (c == 331) opt.sc_ambi = atoi(optarg);
		else if (c == 332) opt.flag |= MM_F_EQX;
		else if (c == 333) opt.flag |= MM_F_PAF_NO_HIT;
		else if (c == 334) opt.split_prefix = optarg;
		else if (c == 335) opt.flag |= MM_F_NO_END_FLT;
		else if (c == 336) opt.flag |= MM_F_HARD_MLEVEL;
		else if (c == 337) opt.max_sw_mat = parse_num(optarg);
		else if (c == 338) opt.max_qlen = (int)parse_num(optarg);
		else if (c == 340) { fprintf(stderr, "[ERROR] --junc-bed belongs to the spliced mode, which this build does not cover\n"); return 1; }
		else if (c == 342) opt.flag |= MM_F_SAM_HIT_ONLY;
		else if (c == 400) n_gpus = atoi(optarg);
		else if (c == 314) yes_or_no(&opt, MM_F_FRAG_MODE, lname, optarg, 1);
		else if (c == 315) yes_or_no(&opt, MM_F_NO_PRINT_2ND, lname, optarg, 0);
		else if (c == 316) { /* --cs */
			opt.flag |= MM_F_OUT_CS | MM_F_CIGAR;
			if (optarg == 0 || strcmp(optarg, "short") == 0) opt.flag &= ~MM_F_OUT_CS_LONG;
			else if (strcmp(optarg, "long") == 0) opt.flag |= MM_F_OUT_CS_LONG;
			else if (strcmp(optarg, "none") == 0) opt.flag &= ~MM_F_OUT_CS;
			else if (mm_verbose >= 2) fprintf(stderr, "[WARNING]\033[1;31m --cs only takes 'short' or 'long'. Invalid values are assumed to be 'short'.\033[0m\n");
		}
		else if (c == 319) yes_or_no(&opt, MM_F_SPLICE_FLANK, lname, optarg, 1);
		else if (c == 324) yes_or_no(&opt, MM_F_HEAP_SORT, lname, optarg, 1);
		else if (c == 326) yes_or_no(&opt, MM_F_NO_DUAL, lname, optarg, 0);
		else if (c == 'S') {
			opt.flag |= MM_F_OUT_CS | MM_F_CIGAR | MM_F_OUT_CS_LONG;
			if (mm_verbose >= 2) fprintf(stderr, "[WARNING]\033[1;31m option -S is deprecated and may be removed in future. Please use --cs=long instead.\033[0m\n");
		} else if (c == 'V') { puts(MM_VERSION); return 0; }
		else if (c == 'f') {
			char *p;
			const double x = strtod(optarg, &p);
			if (x < 1.0) opt.mid_occ_frac = x, opt.mid_occ = 0;
			else opt.mid_occ = (int)(x + .499);
			if (*p == ',') opt.max_occ = (int)(strtod(p + 1, &p) + .499);
		} else if (c == 'u') {
			if (*optarg == 'b') opt.flag |= MM_F_SPLICE_FOR | MM_F_SPLICE_REV;
			else if (*optarg == 'f') opt.flag |= MM_F_SPLICE_FOR, opt.flag &= ~MM_F_SPLICE_REV;
			else if (*optarg == 'r') opt.flag |= MM_F_SPLICE_REV, opt.flag &= ~MM_F_SPLICE_FOR;
			else if (*optarg == 'n') opt.flag &= ~(MM_F_SPLICE_FOR | MM_F_SPLICE_REV);
			else { fprintf(stderr, "[ERROR]\033[1;31m unrecognized cDNA direction\033[0m\n"); return 1; }
		} else if (c == 'z') {
			opt.zdrop = opt.zdrop_inv = strtol(optarg, &s, 10);
			if (*s == ',') opt.zdrop_inv = strtol(s + 1, &s, 10);
		} else if (c == 'O') {
			opt.q = opt.q2 = strtol(optarg, &s, 10);
			if (*s == ',') opt.q2 = strtol(s + 1, &s, 10);
		} else if (c == 'E') {
			opt.e = opt.e2 = strtol(optarg, &s, 10);
			if (*s == ',') opt.e2 = strtol(s + 1, &s, 10);
		}
		longidx = -1;
	}
	if ((opt.flag & MM_F_SPLICE) && (opt.flag & MM_F_FRAG_MODE)) {
		fprintf(stderr, "[ERROR]\033[1;31m --splice and --frag should not be specified at the same time.\033[0m\n");
		return 1;
	}
	if (!fnw && !(opt.flag & MM_F_CIGAR)) ipt.flag |= MM_I_NO_SEQ;
	if (mm_check_opt(&ipt, &opt) < 0) return 1;
	if (opt.best_n == 0) {
		fprintf(stderr, "[WARNING]\033[1;31m changed '-N 0' to '-N %d --secondary=no'.\033[0m\n", old_best_n);
		opt.best_n = old_best_n, opt.flag |= MM_F_NO_PRINT_2ND;
	}
	if (argc == optind || fp_help == stdout) {
		usage(fp_help, &ipt, &opt, n_threads);
		return fp_help == stdout ? 0 : 1;
	}
	if ((opt.flag & MM_F_SR) && argc - optind > 3) {
		fprintf(stderr, "[ERROR] incorrect input: in the sr mode, please specify no more than two query files.\n");
		return 1;
	}
	if (mm_b200_check_opt(&opt) < 0) return 1; /* splice, -D/-X/--dual=no with the sr presets, -T, --split-prefix: refused, not ignored */
	/* two shards per GPU: the host stages (or, for the short-read presets whose bookkeeping runs on the GPU, the upload and
	 * the latency-bound kernel tails) of one overlap the kernels of the other */
	mm_b200_set_lanes(4); /* two lane groups of two streams: two mini-batches in flight on the device path (mm_map_file_frag) */
	if (getenv("MM2_B200_LANES")) mm_b200_set_lanes(atoi(getenv("MM2_B200_LANES")));
	if (mm_b200_set_devices(n_gpus, 0) < 0) { fprintf(stderr, "[ERROR] --gpus must be within 1 and 16\n"); return 1; }
	idx_rdr = mm_idx_reader_open(argv[optind], &ipt, fnw);
	if (idx_rdr == 0) {
		fprintf(stderr, "[ERROR] failed to open file '%s': %s\n", argv[optind], strerror(errno));
		return 1;
	}
	if (!idx_rdr->is_idx && fnw == 0 && argc - optind < 2) {
		fprintf(stderr, "[ERROR] missing input: please specify a query file to map or option -d to keep the index\n");
		mm_idx_reader_close(idx_rdr);
		return 1;
	}
	if (opt.best_n == 0 && (opt.flag & MM_F_CIGAR) && mm_verbose >= 2)
		fprintf(stderr, "[WARNING]\033[1;31m `-N 0' reduces alignment accuracy. Please use --secondary=no to suppress secondary alignments.\033[0m\n");
	while ((mi = mm_idx_reader_read(idx_rdr, n_threads)) != 0) {
		if ((opt.flag & MM_F_OUT_SAM) && idx_rdr->n_parts == 1) {
			if (mm_idx_reader_eof(idx_rdr)) mm_write_sam_hdr(mi, rg, MM_VERSION, argc, argv0);
			else {
				mm_write_sam_hdr(0, rg, MM_VERSION, argc, argv0);
				if (opt.split_prefix == 0 && mm_verbose >= 2)
					fprintf(stderr, "[WARNING]\033[1;31m For a multi-part index, no @SQ lines will be outputted. Please use --split-prefix.\033[0m\n");
			}
		}
		if (mm_verbose >= 3)
			fprintf(stderr, "[M::%s::%.3f*%.2f] loaded/built the index for %d target sequence(s)\n",
					__func__, realtime() - mm_realtime0, cputime() / (realtime() - mm_realtime0), mi->n_seq);
		if (argc != optind + 1) mm_mapopt_update(&opt, mi);
		if (mm_verbose >= 3) mm_idx_stat(mi);
		if (getenv("MM2_B200_PROFILE")) mm_b200_profile(mi, 1);
		if (!(opt.flag & MM_F_FRAG_MODE)) {
			for (i = optind + 1; i < argc; ++i) mm_map_file(mi, argv[i], &opt, n_threads);
		} else mm_map_file_frag(mi, argc - (optind + 1), (const char**)&argv[optind + 1], &opt, n_threads);
		if (mm_verbose >= 4 || getenv("MM2_B200_PROFILE")) mm_b200_report(mi, stderr);
		mm_idx_destroy(mi);
	}
	mm_idx_reader_close(idx_rdr);
	if (fflush(stdout) == EOF) { perror("[ERROR] failed to write the results"); exit(EXIT_FAILURE); }
	if (mm_verbose >= 3) {
		fprintf(stderr, "[M::%s] Version: %s\n", __func__, MM_VERSION);
		fprintf(stderr, "[M::%s] CMD:", __func__);
		for (i = 0; i < argc; ++i) fprintf(stderr, " %s", argv0[i]);
		fprintf(stderr, "\n[M::%s] Real time: %.3f sec; CPU: %.3f sec; Peak RSS: %.3f GB\n", __func__, realtime() - mm_realtime0, cputime(), peakrss() / 1024.0 / 1024.0 / 1024.0);
	}
	return 0;
}
