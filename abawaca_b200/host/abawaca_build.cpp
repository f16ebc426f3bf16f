// abawaca-build (B200): same command line and same output files as the reference program
// (/root/reference/src/abawaca-build.cpp main, :434-634), with the feature stage on the device:
//   SeqIORead_fasta::next_seq       -> abw_fasta_scan / abw_fasta_pack (the FASTA text goes to the device as it is), or for a UCSC .2bit
//                                      file abw_twobit_scan / abw_twobit_pack (the file goes to the device as it is)
//   Scaf::Scaf                      -> abw_segment
//   Scaf_segment::Scaf_segment      -> abw_kmer_features
//   Scaf::add_mapped_read           -> abw_coverage (one call per sample file, reads in file order)
//   SAMReader / ReadMapping(line)   -> abw_parse_sam (SAM text goes to the device in 64 MB chunks cut at line boundaries), or for a BAM file
//                                      abw_bam_feed / abw_bam_finish (the file goes to the device in 64 MB reads, inflated and parsed there)
//   the "%.3lf" rows of abawaca.lrn   -> abw_format_lrn through abwh::write_lrn (text made on the device in 64 MB pieces, written with fwrite)
// The other text writers stay on the host.  Not ported (out of the hot path, SURVEY.md section 2):
// paired-end link counting (abawaca.links is written empty: `abawaca` only checks that it exists) and the calls to
// the external gene predictor / SCG script.
#include "abw_host.h"
#include <algorithm>
#include <ctime>
#include <iostream>
#include <memory>

using namespace abwh;

static std::string stamp()
{
	static time_t t0 = time(nullptr);
	unsigned t = (unsigned)(time(nullptr) - t0);
	char b[32];
	snprintf(b, sizeof(b), "[%02u:%02u:%02u]\t", t / 3600, (t % 3600) / 60, t % 60);
	return b;
}

static void usage(const char* prog)
{
	std::cerr << std::endl << "Usage: " << prog << " -f <fasta-file> -o <out-directory> -s <sam-files-glob> -c <source-sam-file>" << std::endl << std::endl;
}

// the 180 canonical 1..4-mer names in .lrn order: first of {mer, reverse complement} in lexicographic enumeration (abawaca-build.cpp:75-100)
static std::vector<std::string> kmer_names()
{
	std::vector<std::string> names;
	std::map<std::string, size_t> seen;
	for(int k = 1; k <= 4; k++)
		for(int code = 0; code < (1 << (2 * k)); code++) {
			std::string mer(k, 'A'), rc(k, 'A');
			for(int i = 0; i < k; i++) {
				int b = (code >> (2 * (k - 1 - i))) & 3;
				mer[i] = "ACGT"[b];
				rc[k - 1 - i] = "TGCA"[b];
			}
			auto it = seen.find(rc);
			if(it == seen.end()) {
				seen[mer] = names.size();
				names.push_back(mer);
			}
			else
				seen[mer] = it->second;
		}
	return names;
}

static const size_t CHUNK = (size_t)64 << 20;          // bytes per read of a sample file

// the reads of one sample file as device records, in file order
struct SampleReads {
	std::shared_ptr<const abw_read> d_reads;    // its deleter releases the records in the order of the context stream, after what is queued on them
	uint64_t n = 0;
	bool bam = false;
};

// A BAM file goes to the device in CHUNK-byte reads (blocks, header and records may be cut anywhere: the reader carries what is unfinished); SAM
// text in chunks cut at line boundaries, parsed there (abw_parse_sam).  buf: room for CHUNK + 1 bytes, grown for a SAM line longer than that.
static SampleReads sample_reads(abw_ctx* ctx, const abw_names* names, const std::string& path, std::vector<char>& buf)
{
	FILE* fp = fopen(path.c_str(), "rb");
	if(!fp)
		throw std::runtime_error("Failed to open SAM file " + path);
	std::unique_ptr<FILE, int (*)(FILE*)> file(fp, fclose);
	SampleReads out;
	if(is_bgzf(fp)) {
		abw_bam* bam_raw = nullptr;
		ABWH_CHECK(ctx, abw_bam_create(ctx, names, &bam_raw));
		std::unique_ptr<abw_bam, void (*)(abw_bam*)> bam(bam_raw, abw_bam_destroy);
		size_t n;
		while((n = fread(buf.data(), 1, CHUNK, fp)) > 0)
			if(abw_bam_feed(ctx, bam.get(), buf.data(), n) != ABW_OK)
				throw std::runtime_error(std::string("abw_bam_feed failed on ") + path + ": " + abw_last_error(ctx));
		file.reset();
		const abw_read* d_reads = nullptr;
		if(abw_bam_finish(ctx, bam.get(), &d_reads, &out.n) != ABW_OK)
			throw std::runtime_error(std::string("abw_bam_finish failed on ") + path + ": " + abw_last_error(ctx));
		// the records are the reader's: it goes once the device has read them
		out.d_reads = std::shared_ptr<const abw_read>(d_reads, [ctx, b = bam.release()](const abw_read*) { abw_ctx_synchronize(ctx); abw_bam_destroy(b); });
		out.bam = true;
		return out;
	}
	// a record line has at least 11 fields, i.e. at least 10 tabs and a newline: the file size bounds the number of records
	fseek(fp, 0, SEEK_END);
	const uint64_t nlines = (uint64_t)ftell(fp) / 11 + 2;
	rewind(fp);
	abw_read* d_reads = nullptr;
	ABWH_CHECK(ctx, abw_device_alloc(ctx, std::max<uint64_t>(nlines, 1) * sizeof(abw_read), (void**)&d_reads));
	out.d_reads = std::shared_ptr<const abw_read>(d_reads, [ctx](const abw_read* p) { abw_device_free(ctx, (void*)p); });
	size_t have = 0;                                       // bytes of an unfinished line carried over from the previous chunk
	for(;;) {
		if(have == buf.size() - 1)
			buf.resize(2 * buf.size());                    // a line longer than the chunk
		const size_t n = fread(buf.data() + have, 1, buf.size() - 1 - have, fp);
		const size_t total = have + n;
		if(total == 0)
			break;
		size_t cut = total;
		if(n > 0) {                                        // not at the end of the file: cut after the last complete line
			while(cut > 0 && buf[cut - 1] != '\n')
				cut--;
			if(cut == 0) {
				have = total;
				continue;
			}
		}
		uint64_t got = 0;
		int prc = abw_parse_sam(ctx, names, buf.data(), cut, 0, d_reads + out.n, nlines - out.n, &got);
		if(prc == ABW_ERR_ILLEGAL_DNA) {
			std::cerr << "Fatal error, attempted to initialize DNAString with illegal string: " << abw_last_error(ctx) << std::endl;
			exit(-1);
		}
		if(prc != ABW_OK)
			throw std::runtime_error(std::string("abw_parse_sam failed on ") + path + ": " + abw_last_error(ctx));
		out.n += got;
		have = total - cut;
		memmove(buf.data(), buf.data() + cut, have);
		if(n == 0)
			break;
	}
	return out;
}

int main(int argc, const char* argv[])
{
	milestone("start");
	const uint32_t window_size = 2000, max_snps = 15;   // abawaca-build.cpp:436-437
	if(argc < 5) {
		usage(argv[0]);
		return -1;
	}
	std::string assembly_file, out_directory, sam_glob, this_sample_str;
	for(int i = 1; i < argc; i += 2) {
		const char* v = (i + 1 < argc)? argv[i + 1] : "";
		if(!strcmp(argv[i], "-f")) assembly_file = v;
		else if(!strcmp(argv[i], "-o")) out_directory = v;
		else if(!strcmp(argv[i], "-s")) sam_glob = v;
		else if(!strcmp(argv[i], "-c")) this_sample_str = v;
		else {
			std::cerr << std::endl << "Unknown option " << argv[i] << std::endl << std::endl;
			return -1;
		}
	}
	if(assembly_file.empty()) { std::cerr << std::endl << "Error: assembly file was not specified (-f)" << std::endl << std::endl; return -1; }
	if(out_directory.empty()) { std::cerr << std::endl << "Error: output directory was not specified (-o)" << std::endl << std::endl; return -1; }
	if(sam_glob.empty()) { std::cerr << std::endl << "Error: glob path for sam files was not specified (-s)" << std::endl << std::endl; return -1; }
	if(this_sample_str.empty()) { std::cerr << std::endl << "Error: path for sam file for the assembly's reads was not specified (-f)" << std::endl << std::endl; return -1; }

	try {
		std::cerr << stamp() << "Reading assembly file (" << assembly_file << ")" << std::endl;
		abw_ctx* ctx = nullptr;
		if(abw_ctx_create(0, &ctx) != ABW_OK) {
			std::cerr << "Error: no usable CUDA device (abawaca_b200 has no CPU path)" << std::endl;
			return -1;
		}
		milestone("abw_ctx_create");
		// The assembly goes to the device as it is: FASTA text (records indexed there, abw_fasta_scan) or a UCSC .2bit file (decoded there,
		// abw_twobit_pack).  The host only reads the names.
		std::string file_bytes = read_file(assembly_file);
		const bool twobit = is_twobit(file_bytes);
		abw_fasta* fa = nullptr;
		abw_twobit* tb = nullptr;
		if(twobit? abw_twobit_scan(ctx, file_bytes.data(), file_bytes.size(), &tb) != ABW_OK : abw_fasta_scan(ctx, file_bytes.data(), file_bytes.size(), 0, &fa) != ABW_OK)
			throw std::runtime_error(std::string(abw_last_error(ctx)) + " (" + assembly_file + ")");
		const uint64_t nrec = twobit? abw_twobit_count(tb) : abw_fasta_count(fa);
		std::vector<uint64_t> id_off(nrec), rec_len(nrec);
		std::vector<uint32_t> id_len(nrec);
		if(twobit)
			ABWH_CHECK(ctx, abw_twobit_get(ctx, tb, id_off.data(), id_len.data(), rec_len.data()));
		else
			ABWH_CHECK(ctx, abw_fasta_get(ctx, fa, id_off.data(), id_len.data(), rec_len.data()));
		// scaffolds in name order; the first record of a name wins (std::map::insert, abawaca-build.cpp:482-490)
		std::map<std::string, size_t> by_name;
		for(size_t i = 0; i < nrec; i++) {
			if(rec_len[i] == 0)
				std::cerr << "Warning: sequence " << file_bytes.substr(id_off[i], id_len[i]) << " is empty" << std::endl;      // SeqIORead_fasta.h:99-101
			by_name.insert(std::make_pair(file_bytes.substr(id_off[i], id_len[i]), i));
		}
		const uint32_t nscaf = (uint32_t)by_name.size();
		std::vector<std::string> scaf_name;
		std::vector<uint64_t> scaf_len;
		std::vector<uint32_t> order;
		for(auto& kv : by_name) {
			scaf_name.push_back(kv.first);
			scaf_len.push_back(rec_len[kv.second]);
			order.push_back((uint32_t)kv.second);
		}
		abw_seqset* ss = nullptr;
		int rc;
		if(twobit) {
			void* d_file = nullptr;
			ABWH_CHECK(ctx, abw_device_alloc(ctx, std::max<size_t>(file_bytes.size(), 1), &d_file));
			ABWH_CHECK(ctx, abw_copy_to_device(ctx, d_file, file_bytes.data(), file_bytes.size()));
			rc = abw_twobit_pack(ctx, tb, d_file, 0, order.data(), nscaf, &ss);
			ABWH_CHECK(ctx, abw_ctx_synchronize(ctx));
			ABWH_CHECK(ctx, abw_device_free(ctx, d_file));
			abw_twobit_destroy(tb);
		}
		else {
			rc = abw_fasta_pack(ctx, fa, order.data(), nscaf, &ss);
			abw_fasta_destroy(fa);
		}
		std::string().swap(file_bytes);
		if(rc != ABW_OK) {
			std::cerr << "Fatal error, attempted to initialize DNAString with illegal string: " << abw_last_error(ctx) << std::endl;
			return -1;
		}
		abw_segments* sg = nullptr;
		ABWH_CHECK(ctx, abw_segment(ctx, ss, window_size, &sg));
		const uint64_t ndps = abw_segments_count(sg);
		milestone("FASTA");

		if(!directory_exists(out_directory)) {
			std::string cmd = "mkdir " + out_directory;
			if(system(cmd.c_str()) != 0)
				std::cerr << "Warning: could not create " << out_directory << std::endl;
		}
		const std::string names_file = out_directory + "/abawaca.names", lrn_file = out_directory + "/abawaca.lrn", info_file = out_directory + "/abawaca.info",
		                  links_file = out_directory + "/abawaca.links";
		std::cerr << stamp() << "Creating .lrn (" << lrn_file << ") and .names (" << names_file << ") files" << std::endl;

		const std::vector<std::string> sam_files = glob_files(sam_glob);
		const uint64_t ld = 179 + sam_files.size();
		double* d_rows = nullptr;
		uint64_t* d_nbps = nullptr;
		ABWH_CHECK(ctx, abw_device_alloc(ctx, std::max<uint64_t>(ndps * ld, 1) * sizeof(double), (void**)&d_rows));
		ABWH_CHECK(ctx, abw_device_alloc(ctx, std::max<uint32_t>(nscaf, 1) * sizeof(uint64_t), (void**)&d_nbps));
		ABWH_CHECK(ctx, abw_memset_device(ctx, d_nbps, 0, std::max<uint32_t>(nscaf, 1) * sizeof(uint64_t)));
		ABWH_CHECK(ctx, abw_kmer_features(ctx, ss, sg, ABW_FEAT_TRUNC3, 1, d_rows, ld, 0));
		ABWH_CHECK(ctx, abw_ctx_synchronize(ctx));
		milestone("k-mer");

		// the scaffold names as a device-side table: SAM text is parsed on the device (abw_parse_sam)
		abw_names* names = nullptr;
		{
			std::string blob;
			std::vector<uint64_t> noff(1, 0);
			for(auto& kv : by_name) {
				blob += kv.first;
				noff.push_back(blob.size());
			}
			ABWH_CHECK(ctx, abw_names_create(ctx, blob.data(), noff.data(), nscaf, &names));
		}
		std::vector<char> buf(CHUNK + 1);
		for(size_t j = 0; j < sam_files.size(); j++) {
			std::cerr << stamp() << "Reading SAM file " << sam_files[j] << std::endl;
			const bool is_this_sample = (sam_files[j] == this_sample_str);
			SampleReads reads = sample_reads(ctx, names, sam_files[j], buf);
			ABWH_CHECK(ctx, abw_coverage(ctx, sg, reads.d_reads.get(), reads.n, 1, max_snps, ABW_FEAT_TRUNC3, d_rows, ld, (uint32_t)(179 + j),
			                             is_this_sample? d_nbps : nullptr));
			reads.d_reads.reset();
			milestone((reads.bam? "BAM " : "SAM ") + std::to_string(j));
			if(is_this_sample) {
				FILE* fl = fopen(links_file.c_str(), "w");     // scaffold-end links are not computed (SURVEY.md section 2, row 5); the file must exist
				if(fl) fclose(fl);
			}
		}
		abw_names_destroy(names);

		// fetch what .names and .info need (the matrix stays on the device: abw_format_lrn prints it)
		std::vector<uint32_t> seg_scaf(ndps);
		std::vector<uint64_t> seg_start(ndps), seg_end(ndps), seg_nonN(ndps), nbps(nscaf), nN(nscaf), nGC(nscaf);
		ABWH_CHECK(ctx, abw_segments_get(ctx, sg, nullptr, seg_scaf.data(), seg_start.data(), seg_end.data(), seg_nonN.data()));
		if(nscaf)
			ABWH_CHECK(ctx, abw_copy_to_host(ctx, nbps.data(), d_nbps, nscaf * sizeof(uint64_t)));
		ABWH_CHECK(ctx, abw_seqset_stats(ctx, ss, nN.data(), nGC.data()));
		milestone("fetch");

		FILE* fout = fopen(names_file.c_str(), "w");
		FILE* flrn = fopen(lrn_file.c_str(), "w");
		FILE* finfo = fopen(info_file.c_str(), "w");
		if(!fout) { std::cerr << "Could not write to " << names_file << std::endl << std::endl; return -1; }
		if(!flrn) { std::cerr << "Could not write to " << lrn_file << std::endl << std::endl; return -1; }
		if(!finfo) { std::cerr << "Could not write to " << info_file << std::endl << std::endl; return -1; }
		fprintf(fout, "%c %lu\n", '%', (unsigned long)ndps);
		{
			// the columns: the k-mers but the first ("A", which the reference does not write) and one per sample; "%.3lf" values
			std::vector<std::string> cols = kmer_names();
			cols.erase(cols.begin());
			cols.insert(cols.end(), sam_files.begin(), sam_files.end());
			char* d_text = nullptr;
			ABWH_CHECK(ctx, abw_device_alloc(ctx, LRN_CHUNK, (void**)&d_text));
			std::vector<char> text;
			if(!write_lrn(ctx, flrn, cols, d_rows, ld, nullptr, ndps, ABW_TEXT_3LF, d_text, text)) { std::cerr << "Could not write to " << lrn_file << std::endl << std::endl; return -1; }
			ABWH_CHECK(ctx, abw_device_free(ctx, d_text));
		}
		fclose(flrn);
		milestone(".lrn");
		uint64_t g = 0;
		for(uint32_t s = 0; s < nscaf; s++) {
			const std::string& id = scaf_name[s];
			const double len = (double)scaf_len[s];
			const double cvg = (double)nbps[s] / len;
			const double denom = len - (double)nN[s];
			const double gc = (denom == 0)? 0 : (double)nGC[s] / denom;
			fprintf(finfo, "%s\t%lu\t%.3lf\t%.3lf\t%lu\n", id.c_str(), (unsigned long)scaf_len[s], int(1000.0 * cvg) / 1000.0, int(1000.0 * gc) / 1000.0,
			        (unsigned long)nN[s]);
			unsigned long k = 0;
			for(; g < ndps && seg_scaf[g] == s; g++) {
				k++;
				fprintf(fout, "%lu\t%s_%lu\t%s:(%lu, %lu), %lu/%lu non-Ns bps\n", (unsigned long)(g + 1), id.c_str(), k, id.c_str(), (unsigned long)seg_start[g],
				        (unsigned long)seg_end[g], (unsigned long)seg_nonN[g], (unsigned long)(seg_end[g] - seg_start[g] + 1));
			}
		}
		fclose(fout);
		fclose(finfo);
		milestone(".names, .info");

		std::cerr << stamp() << "Predicting genes and SCGs (skipped: external tools are not part of this build; pass -c <gene2scg> to abawaca)" << std::endl;
		size_t l = assembly_file.rfind('/');
		const std::string out_name = (l == std::string::npos)? assembly_file : assembly_file.substr(l + 1);
		const std::string scg_file = out_directory + "/" + out_name + ".proteins.faa.bacteria.scg";
		const std::string data = out_directory + "/data.txt";
		FILE* fp = fopen(data.c_str(), "w");
		if(!fp) { std::cerr << "Could not write to " << data << std::endl << std::endl; return -1; }
		{
		// the reference's prepare_scgs leaves this file behind (abawaca-build.cpp:401-431); without the external gene caller it is created empty so that
		// the two-step command line (abawaca-build, then abawaca -u DIR -o OUT) runs: no SCG information unless abawaca gets -c <gene2scg>
		FILE* fs = fopen(scg_file.c_str(), "a");
		if(fs) fclose(fs);
	}
	fprintf(fp, "SCG\t%s\n", scg_file.c_str());
		fprintf(fp, "Links\t%s\n", links_file.c_str());
		fprintf(fp, "Info\t%s\n", info_file.c_str());
		fprintf(fp, "Names\t%s\n", names_file.c_str());
		fprintf(fp, "Lrn\t%s\n", lrn_file.c_str());
		fprintf(fp, "Assembly\t%s\n", assembly_file.c_str());
		fclose(fp);

		abw_device_free(ctx, d_rows);
		abw_device_free(ctx, d_nbps);
		abw_segments_destroy(sg);
		abw_seqset_destroy(ss);
		abw_ctx_destroy(ctx);
		milestone("teardown");
		std::cerr << stamp() << "Finished successfully" << std::endl;
	}
	catch(std::exception& e) {
		std::cerr << "Fatal error: " << e.what() << std::endl;
		return -1;
	}
	return 0;
}
