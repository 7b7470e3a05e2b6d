// What the two FASTQ readers share: the host reader cls_fastq_read (record_writer.cpp) and the device ingest
// cls_fastq_upload (capi.cu, fastq_kernels.cu) refuse a malformed file with the same first bad record and reason.
#pragma once
#include <cstdint>

namespace cls {

// Why a record is malformed, in the order the checks of one record run (its first failing check is its reason).
enum FastqReason : int {
    kFastqBlankLine = 1,      // a blank title line with records after it
    kFastqNoAt = 2,           // the title line does not start with '@'
    kFastqTruncated = 3,      // fewer than four lines left
    kFastqNoPlus = 4,         // the separator line does not start with '+'
    kFastqQualityLength = 5,  // the quality line's length differs from the sequence line's
    kFastqTitleUtf8 = 6,      // the title is not valid UTF-8
};

const char *fastq_reason(int code);
// Sets "malformed FASTQ record <record + 1>: <reason>" and returns CLS_ERR_INVALID_ARGUMENT.
int fastq_fail(uint64_t record, int code);
// Number of records of a text with `n_newlines` newlines: the lines up to the last non-blank one, four per record (the last
// one possibly truncated).
uint64_t fastq_n_records(const uint8_t *text, uint64_t n, uint64_t n_newlines);
// First record r < n_records whose title text[hb[r] .. he[r]) is not valid UTF-8, or n_records (on the host pool).
uint64_t fastq_first_bad_title(const uint8_t *text, const uint64_t *hb, const uint64_t *he, uint64_t n_records);

}  // namespace cls
