#!/usr/bin/env python
'''
Mirror of the reference's runGan.py launcher (run cases, reference runGan.py:1-10):
python3 runGan.py 1   # inference on LR/calendar with the flags of record (reference runGan.py:67-90)
python3 runGan.py 3   # train TecoGAN  (reference runGan.py:107-244)
python3 runGan.py 4   # train FRVSR    (reference runGan.py:247-296)
python3 runGan.py 2   # PSNR / SSIM of ./results/<scene> against ./HR/<scene> on the GPU (reference runGan.py:92-105; tOF
                      # is available through `metrics.py --keys PSNR,SSIM,tOF`; LPIPS / tLP are not, DESIGN.md section 6)
Case 0 (download, needs network) is outside the hot path and prints why it is not run.
Extra arguments after the case number are appended to the main.py command line (e.g. --max_iter 100).
'''
import datetime
import os
import signal
import subprocess
import sys

runcase = int(sys.argv[1]) if len(sys.argv) > 1 else 1
extra = sys.argv[2:]
print("Testing test case %d" % runcase)
HERE = os.path.dirname(os.path.abspath(__file__))
MAIN = os.path.join(HERE, "main.py")


def preexec():  # Don't forward signals.
    os.setpgrp()


def mycall(cmd, block=False):
    return subprocess.Popen(cmd, preexec_fn=preexec) if block else subprocess.Popen(cmd)


def run_train(cmd1):
    pid = mycall(cmd1, block=True)
    try:
        pid.communicate()
    except KeyboardInterrupt:   # reference runGan.py:237-244
        print("runGAN.py: sending SIGINT signal to the sub process...")
        pid.send_signal(signal.SIGINT)
        pid.communicate()
        print("runGAN.py: finished...")


TrainingDataPath = os.environ.get("TECO_TRAINING_DATA", "/mnt/netdisk/video_data/")   # reference runGan.py:135,274: "update the TrainingDataPath"

if runcase == 0:
    print("case 0 downloads models/data with wget (reference runGan.py:41-65); there is no network here.")
elif runcase == 1:   # inference a trained model
    dirstr = './results/'
    testpre = ['calendar']
    os.makedirs(dirstr, exist_ok=True)
    lr_root = "./LR/" if os.path.exists("./LR/") else "/root/reference/LR/"
    # reference runGan.py:87: --checkpoint ./model/TecoGAN (a TF V2 bundle, read without TensorFlow); then our .pt; else seeded init
    ckpt = ('./model/TecoGAN' if os.path.exists('./model/TecoGAN.index') else
            './model/TecoGAN.pt' if os.path.exists('./model/TecoGAN.pt') else 'random:1234')
    for nn in range(len(testpre)):
        cmd1 = [sys.executable, MAIN, "--cudaID", "0", "--output_dir", dirstr, "--summary_dir", os.path.join(dirstr, 'log/'),
                "--mode", "inference", "--input_dir_LR", os.path.join(lr_root, testpre[nn]), "--output_pre", testpre[nn],
                "--num_resblock", "16", "--checkpoint", ckpt, "--output_ext", "png"] + extra
        mycall(cmd1).communicate()
elif runcase == 2:
    testpre = ["calendar"]                       # reference runGan.py:94-105
    dirstr, tarstr = './results/', './HR/'
    cmd1 = [sys.executable, os.path.join(HERE, "metrics.py"), "--output", dirstr + "metric_log/",
            "--results", ",".join(dirstr + _ for _ in testpre), "--targets", ",".join(tarstr + _ for _ in testpre)] + extra
    mycall(cmd1).communicate()
elif runcase == 3:   # Train TecoGAN -- flags of record reference runGan.py:142-234
    now_str = datetime.datetime.now().strftime("%m-%d-%H")
    train_dir = "ex_TecoGAN%s/" % now_str
    cmd1 = [sys.executable, MAIN, "--cudaID", "0", "--output_dir", train_dir, "--summary_dir", os.path.join(train_dir, "log/"),
            "--mode", "train", "--batch_size", "4", "--RNN_N", "10", "--movingFirstFrame", "--random_crop", "--crop_size", "32",
            "--input_video_dir", TrainingDataPath, "--input_video_pre", "scene", "--str_dir", "2000", "--end_dir", "2250",
            "--end_dir_val", "2290", "--max_frm", "119", "--queue_thread", "12",   # reference runGan.py:178-184 / 276-282
            "--learning_rate", "0.00005", "--decay_step", "500000", "--decay_rate", "1.0", "--stair", "--beta", "0.9",
            "--max_iter", "500000", "--save_freq", "10000", "--num_resblock", "16", "--vgg_scaling", "0.2",
            "--ratio", "0.01", "--Dt_mergeDs", "--Dt_ratio_max", "1.0", "--Dt_ratio_0", "1.0", "--Dt_ratio_add", "0.0",
            "--pingpang", "--pp_scaling", "0.5", "--D_LAYERLOSS"] + extra
    if os.path.exists('./model/vgg_19.ckpt'):            # reference runGan.py:113-115,176
        cmd1 += ["--vgg_ckpt", './model/vgg_19.ckpt']
    if os.path.exists('./model/ourFRVSR.index'):         # reference runGan.py:121-133,201-207: start from the FRVSR weights
        cmd1 += ["--pre_trained_model", "--checkpoint", './model/ourFRVSR']
    run_train(cmd1)
elif runcase == 4:   # Train FRVSR -- flags of record reference runGan.py:250-286
    now_str = datetime.datetime.now().strftime("%m-%d-%H")
    train_dir = "ex_FRVSR%s/" % now_str
    cmd1 = [sys.executable, MAIN, "--cudaID", "0", "--output_dir", train_dir, "--summary_dir", os.path.join(train_dir, "log/"),
            "--mode", "train", "--batch_size", "4", "--RNN_N", "10", "--movingFirstFrame", "--random_crop", "--crop_size", "32",
            "--input_video_dir", TrainingDataPath, "--input_video_pre", "scene", "--str_dir", "2000", "--end_dir", "2250",
            "--end_dir_val", "2290", "--max_frm", "119", "--queue_thread", "12",   # reference runGan.py:178-184 / 276-282
            "--learning_rate", "0.00005", "--decay_step", "500000", "--decay_rate", "1.0", "--stair", "--beta", "0.9",
            "--max_iter", "500000", "--save_freq", "10000", "--num_resblock", "10", "--ratio", "-0.01", "--nopingpang"] + extra
    run_train(cmd1)
