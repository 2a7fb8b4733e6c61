/*
 * oracle/dropin_harness.c — TEST INFRASTRUCTURE ONLY (never linked into libvdl2gpu.so).
 *
 * A stand-in for the dumpvdl2 program around libvdl2gpu.so's drop-in symbols (include/vdl2_dropin.h): it drives them
 * with the reference's init / feed protocol, as oracle/ref_harness.c drives the reference's own demodulator
 *   vdl2_channel_init xN, rs_init, *_init, sbuf, two barriers of N+1, one process_samples pthread per channel,
 *   process_buf_* per chunk, the final wait on demods_ready                       (reference src/dumpvdl2.c:1086-1170)
 * and supplies what the rest of dumpvdl2 would: the globals `demods_ready`, `samples_ready` and the upper boundary
 * avlc_decoder_queue_push(), which here captures (metadata, frame) per channel instead of queueing them for the AVLC
 * decoder thread (reference src/decode.c:165-171; the consumer owns and frees all three allocations).
 *
 * Usage: dropin_harness --fmt u8|s16 --oversample N --centerfreq HZ --freqs f0,f1,... [--chunk BYTES] FILE
 * Output (stdout), the format of oracle/ref_harness.c: one line per pushed frame, sorted by (channel, push order):
 *   FRAME ch=I freq=F idx=K len=L synd=W datalen=D fec=C pwr=%.9g nf=%.9g ppm=%.9g hex=...
 */
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>
#include "vdl2_dropin.h"

pthread_barrier_t demods_ready, samples_ready;

typedef struct captured {
	vdl2_msg_metadata md;
	uint8_t *buf;
	size_t len;
	struct captured *next;
} captured_t;

static struct { captured_t *head, *tail; } *captures;
static uint32_t *chan_freqs;
static int num_channels;
static pthread_mutex_t capture_lock = PTHREAD_MUTEX_INITIALIZER;

/* The drop-in pushes every channel's frames from one thread: the channel is the first one on the frame's frequency. */
void avlc_decoder_queue_push(vdl2_msg_metadata *metadata, octet_string_t *frame, int flags) {
	(void)flags;
	int chan = 0;
	while(chan < num_channels && chan_freqs[chan] != metadata->freq) chan++;
	if(chan == num_channels) { fprintf(stderr, "frame for an unknown frequency %u\n", metadata->freq); _exit(4); }
	captured_t *c = calloc(1, sizeof(*c));
	c->md = *metadata;
	c->buf = frame->buf;
	c->len = frame->len;
	pthread_mutex_lock(&capture_lock);
	if(captures[chan].tail) captures[chan].tail->next = c; else captures[chan].head = c;
	captures[chan].tail = c;
	pthread_mutex_unlock(&capture_lock);
	free(frame);
	free(metadata);
}

static void *chan_thread(void *arg) { return process_samples(arg); }

int main(int argc, char **argv) {
	char const *fmt = "u8", *freqs_s = NULL, *file = NULL;
	uint32_t oversample = 10, centerfreq = 0, chunk = 320000;
	for(int i = 1; i < argc; i++) {
		if(!strcmp(argv[i], "--fmt") && i + 1 < argc) fmt = argv[++i];
		else if(!strcmp(argv[i], "--oversample") && i + 1 < argc) oversample = strtoul(argv[++i], NULL, 10);
		else if(!strcmp(argv[i], "--centerfreq") && i + 1 < argc) centerfreq = strtoul(argv[++i], NULL, 10);
		else if(!strcmp(argv[i], "--freqs") && i + 1 < argc) freqs_s = argv[++i];
		else if(!strcmp(argv[i], "--chunk") && i + 1 < argc) chunk = strtoul(argv[++i], NULL, 10);
		else if(argv[i][0] != '-') file = argv[i];
		else { fprintf(stderr, "unknown option %s\n", argv[i]); return 2; }
	}
	if(!file || !freqs_s || chunk == 0) { fprintf(stderr, "need --freqs and FILE\n"); return 2; }
	int is_s16 = !strcmp(fmt, "s16");
	char *dup = strdup(freqs_s), *save = NULL;
	for(char *t = strtok_r(dup, ",", &save); t; t = strtok_r(NULL, ",", &save)) {
		chan_freqs = realloc(chan_freqs, (num_channels + 1) * sizeof(uint32_t));
		chan_freqs[num_channels++] = strtoul(t, NULL, 10);
	}
	free(dup);
	if(num_channels == 0) { fprintf(stderr, "empty --freqs\n"); return 2; }
	if(centerfreq == 0) centerfreq = chan_freqs[0];
	uint32_t sample_rate = 105000 * oversample;          /* SYMBOL_RATE * SPS * oversample, reference src/dumpvdl2.c:1073 */

	FILE *f = fopen(file, "rb");
	if(!f) { perror(file); return 2; }
	fseek(f, 0, SEEK_END);
	long fsize = ftell(f);
	fseek(f, 0, SEEK_SET);
	unsigned char *data = malloc(fsize ? fsize : 1);
	if(fread(data, 1, fsize, f) != (size_t)fsize) { perror("fread"); return 2; }
	fclose(f);

	captures = calloc(num_channels, sizeof(*captures));
	vdl2_channel_t **chans = calloc(num_channels, sizeof(*chans));
	for(int i = 0; i < num_channels; i++)
		chans[i] = vdl2_channel_init(centerfreq, chan_freqs[i], sample_rate, oversample);
	if(rs_init() < 0) { fprintf(stderr, "rs_init failed\n"); return 3; }
	sincosf_lut_init();
	input_lpf_init(sample_rate);
	demod_sync_init();
	process_buf_uchar_init();
	sbuf = calloc(chunk, sizeof(float));
	pthread_barrier_init(&demods_ready, NULL, num_channels + 1);
	pthread_barrier_init(&samples_ready, NULL, num_channels + 1);
	for(int i = 0; i < num_channels; i++)
		pthread_create(&chans[i]->demod_thread, NULL, chan_thread, chans[i]);

	for(long off = 0; off < fsize; off += chunk) {
		uint32_t len = (uint32_t)((fsize - off) < (long)chunk ? (fsize - off) : (long)chunk);
		if(is_s16) process_buf_short(data + off, len, NULL);
		else process_buf_uchar(data + off, len, NULL);
	}
	pthread_barrier_wait(&demods_ready);                  /* drain: reference src/dumpvdl2.c:1170 */
	if(vdl2gpu_dropin_last_status() != 0) { fprintf(stderr, "drop-in status %d\n", vdl2gpu_dropin_last_status()); _exit(5); }

	for(int i = 0; i < num_channels; i++) {
		for(captured_t *c = captures[i].head; c; c = c->next) {
			printf("FRAME ch=%d freq=%u idx=%d len=%zu synd=%u datalen=%u fec=%d pwr=%.9g nf=%.9g ppm=%.9g hex=",
					i, c->md.freq, c->md.idx, c->len, c->md.synd_weight, c->md.datalen_octets,
					c->md.num_fec_corrections, c->md.frame_pwr_dbfs, c->md.nf_pwr_dbfs, c->md.ppm_error);
			for(size_t k = 0; k < c->len; k++) printf("%02x", c->buf[k]);
			printf("\n");
		}
	}
	fflush(stdout);
	_exit(0);   /* channel threads are parked on the barrier; no join (same as the reference's shutdown) */
}
